// Weight gradient of a pointwise channel map on the tensor cores (tcgen05 / TMEM, 3xTF32):
//     dW[o][c] = sum over (batch, voxel) of dy[o][v] x[c][v],   db[o] = sum of dy[o][v]
// (reference factorizer/layers/linear.py:53-58: a k = 1 Conv1d; the wide blocks' linears, the patch convolutions on their
// space-to-depth view, the stem on its unfolded input).
//
// A contraction over voxels of two operands that lie in memory exactly as the tensor core wants a K-major operand:
// rows = channels, K = voxels, contiguous.  TMA brings a (64 channels x 32 voxels) box of dy and of x per stage straight into
// the SWIZZLE_128B layout; that fp32 tile is the "hi" operand as it stands (the tensor core reads the top 19 bits of a word).
// Four warps compute the remainder tiles lo = v - hi(v) element by element (same shared-memory offsets, so the swizzle is
// never decoded), and ONE MMA per 8 voxels with A = [dy ; dy_lo] (M = 128) and B = [x ; x_lo ; ones] (N = 144) produces all
// four hi / lo blocks of a 64 x 64 block of dW plus the bias column; they accumulate in TMEM over the CTA's share of the
// voxels and are added up, then added to the global gradient with one atomic per element and CTA (the chain is capped at
// cmap::wgrad_ctas's 32 stages per CTA).
// Warp roles: warp 0 = TMA producer, warp 1 = MMA issue (warp-uniform code under elect.sync), warps 2-5 = remainder tiles and
// epilogue.  Three stages of 32 KB, two CTAs per SM.
#include "fz_channel_map.cuh"
#include "fz_tc.cuh"

namespace fz {
namespace {

using namespace tc;

constexpr int kBlk = 64;                       // channels per block of dW, both ways
constexpr int kVT = 32;                        // voxels per stage = one 128-byte swizzle row
constexpr int kStages = 3;
constexpr int kThreads = 192;
constexpr uint32_t kTile = kBlk * 128;         // one (64 x 32) fp32 tile: 8 KiB
// stage: dy hi | dy lo | x hi | x lo | ones block (16 rows: the first all ones)
constexpr uint32_t oA = 0, oB = 2 * kTile, oOnes = 4 * kTile, kStage = 4 * kTile + 16 * 128;
constexpr uint32_t oBarFull = kStages * kStage, oBarLo = oBarFull + 8 * kStages, oBarEmpty = oBarLo + 8 * kStages,
                   oBarDone = oBarEmpty + 8 * kStages, oTmemSlot = oBarDone + 8, kSmemW = oTmemSlot + 8;
constexpr int kN = 2 * kBlk + 16;              // 144 accumulator columns

// (batch, channels, voxels) fp32, box (1, 64, 32): rows beyond `channels` read as zeros, so do voxels beyond the end
int make_map(CUtensorMap* m, const float* ptr, long long batch, int channels, long long voxels) {
    cuuint64_t dims[3] = {(cuuint64_t)voxels, (cuuint64_t)channels, (cuuint64_t)batch};
    cuuint64_t strides[2] = {(cuuint64_t)voxels * 4, (cuuint64_t)voxels * channels * 4};
    cuuint32_t box[3] = {kVT, kBlk, 1};
    return encode_tiled_map(m, "dy / x", CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, ptr, dims, strides, box,
                            CU_TENSOR_MAP_SWIZZLE_128B);
}

__global__ void __launch_bounds__(kThreads, 2)
linear_wgrad_tc(const __grid_constant__ CUtensorMap map_dy, const __grid_constant__ CUtensorMap map_x, float* __restrict__ dW,
                float* __restrict__ db, int cout, int cin, int tiles_per_sample, long long total_tiles) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const uint32_t sbase = smem_u32(smem);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = (int)uniform_u32((uint32_t)(tid >> 5));
    const int ob = blockIdx.y, ib = blockIdx.z;
    const long long my_tiles = blockIdx.x < total_tiles ? (total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(sbase + oBarFull + 8 * s, 1);
            mbar_init(sbase + oBarLo + 8 * s, 4);
            mbar_init(sbase + oBarEmpty + 8 * s, 1);
        }
        mbar_init(sbase + oBarDone, 1);
        fence_mbarrier_init();
    }
    // the ones block of every stage (constant): row 0 = ones, rows 1 .. 15 = zeros (a 128-byte row of equal words: no swizzle to mind)
    for (int i = tid; i < kStages * 16 * 32; i += kThreads) {
        const int s = i / (16 * 32), r = (i / 32) % 16;
        reinterpret_cast<float*>(smem + s * kStage + oOnes)[i % (16 * 32)] = r == 0 ? 1.f : 0.f;
    }
    if (warp == 1) {
        tmem_alloc<256>(sbase + oTmemSlot);
        tmem_relinquish_alloc_permit();
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = uniform_u32(*reinterpret_cast<const uint32_t*>(smem + oTmemSlot));

    if (warp == 0) {
        // ---- TMA producer ----
        if (elect_one()) {
            long long nb = (long long)blockIdx.x / tiles_per_sample;
            int nt = (int)((long long)blockIdx.x - nb * tiles_per_sample);
            for (long long it = 0; it < my_tiles; ++it) {
                const int s = (int)(it % kStages);
                const uint32_t round = (uint32_t)(it / kStages);
                if (round > 0) mbar_wait(sbase + oBarEmpty + 8 * s, (round - 1) & 1);
                const uint32_t full = sbase + oBarFull + 8 * s;
                mbar_arrive_expect_tx(full, 2 * kTile);
                tma_load_3d(sbase + s * kStage + oA, &map_dy, full, nt * kVT, ob * kBlk, (int)nb);
                tma_load_3d(sbase + s * kStage + oB, &map_x, full, nt * kVT, ib * kBlk, (int)nb);
                nt += (int)gridDim.x;
                while (nt >= tiles_per_sample) { nt -= tiles_per_sample; ++nb; }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ---- MMA issue: D[128 x 144] += [dy ; dy_lo] (rows) x [x ; x_lo ; ones] (columns) over the stage's 4 groups of 8 voxels ----
        const uint32_t idesc = make_idesc(128, kN, false, false);
        for (long long it = 0; it < my_tiles; ++it) {
            const int s = (int)(it % kStages);
            const uint32_t round = (uint32_t)(it / kStages);
            mbar_wait(sbase + oBarLo + 8 * s, round & 1);
            tc_fence_after();
            if (elect_one()) {
                const uint64_t ad = make_desc(sbase + s * kStage + oA, 16, 1024, 2);
                const uint64_t bd = make_desc(sbase + s * kStage + oB, 16, 1024, 2);
#pragma unroll
                for (int k = 0; k < kVT / 8; ++k) mma_tf32(tmem, desc_at(ad, k * 32), desc_at(bd, k * 32), idesc, it > 0 || k > 0);
                commit(sbase + oBarEmpty + 8 * s);
                if (it + 1 == my_tiles) commit(sbase + oBarDone);
            }
            __syncwarp();
        }
    } else {
        // ---- remainder tiles: lo = v - hi(v), word by word at the same shared-memory offsets ----
        const int t = tid - 64;                                // 0 .. 127
        for (long long it = 0; it < my_tiles; ++it) {
            const int s = (int)(it % kStages);
            const uint32_t round = (uint32_t)(it / kStages);
            mbar_wait(sbase + oBarFull + 8 * s, round & 1);
            unsigned char* st = smem + s * kStage;
#pragma unroll
            for (int half = 0; half < 2; ++half) {             // dy tile, then x tile
                const float4* hi = reinterpret_cast<const float4*>(st + (half ? oB : oA));
                float4* lo = reinterpret_cast<float4*>(st + (half ? oB : oA) + kTile);
#pragma unroll
                for (int i = 0; i < (int)(kTile / 16) / 128; ++i) {
                    const float4 v = hi[i * 128 + t];
                    lo[i * 128 + t] = make_float4(tf32_lo(v.x), tf32_lo(v.y), tf32_lo(v.z), tf32_lo(v.w));
                }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(sbase + oBarLo + 8 * s);
        }
    }
    // ---- epilogue: accumulator row r (TMEM lane r) = output channel r % 64 (hi block for r < 64, lo block above); column n =
    //      input channel n % 64 (hi for n < 64, lo for 64 <= n < 128), column 128 = the bias sums ----
    if (my_tiles > 0) {
        mbar_wait(sbase + oBarDone, 0);
        tc_fence_after();
    }
    __syncthreads();                                           // the stages are free: they take the scratch copy of the accumulator
    float* S = reinterpret_cast<float*>(smem);                 // [128][145]
    if (my_tiles > 0 && warp >= 2) {
        const int q = warp & 3;                                // the TMEM lane quarter this warp may read
        const int r = q * 32 + lane;
        const uint32_t row_addr = tmem + ((uint32_t)(q * 32) << 16);
#pragma unroll
        for (int c0 = 0; c0 < 128; c0 += 32) {
            float d[32];
            tmem_ld32(row_addr + c0, d);
#pragma unroll
            for (int c = 0; c < 32; ++c) S[r * 145 + c0 + c] = d[c];
        }
        uint32_t e[16];
        tmem_ld16_nowait(row_addr + 128, e);
        tmem_ld_wait();
        S[r * 145 + 128] = __uint_as_float(e[0]);
    }
    tc_fence_before();
    __syncthreads();
    if (my_tiles > 0) {
        for (int i = tid; i < kBlk * kBlk; i += kThreads) {
            const int o = i >> 6, c = i & 63;
            const int go = ob * kBlk + o, gc = ib * kBlk + c;
            if (go < cout && gc < cin) {
                const float v = (S[o * 145 + c] + S[o * 145 + 64 + c]) + (S[(64 + o) * 145 + c] + S[(64 + o) * 145 + 64 + c]);
                atomicAdd(dW + (size_t)go * cin + gc, v);
            }
        }
        if (db && ib == 0 && tid < kBlk && ob * kBlk + tid < cout) atomicAdd(db + ob * kBlk + tid, S[tid * 145 + 128] + S[(64 + tid) * 145 + 128]);
    }
    __syncthreads();
    if (warp == 1) tmem_dealloc<256>(tmem);
}

// =====================================================================================================================
// y[b][o][v] = sum_c W[o][c] x[b][c][v] (+ bias[o]): the channel map itself, any channel counts (the wide blocks' linears and
// MLPs, the patch convolutions on their space-to-depth view; with W^T it is the input gradient).  3xTF32 on tcgen05:
//   D[128 voxels x 64 outputs] += A[128 x 32 channels] B[64 x 32]^T per K chunk,
// A = x, voxel-contiguous = MN-major: TMA boxes of (32 channels x 32 voxels) with SWIZZLE_128B_ATOM_32B are exactly the atoms
// of the one swizzle 32-bit MN-major operands accept; B = W, K-major, SWIZZLE_128B boxes as in the weight-gradient kernel.
// The fp32 tiles are the hi operands; eight warps write the remainder tiles and later run the epilogue (cmap::Epilogue in
// fz_channel_map.cuh, shared with the bf16 channel map: thread = voxel = TMEM lane; bias / residual loaded into the running
// sums an item ahead; FZ_EPILOGUE_*: + residual, GELU, GELU derivative; coalesced stores along the voxel axis).  Persistent
// CTAs walk (voxel tile, output tile) items; K chunks flow through a two-stage (four-stage for launches with fewer items than
// SMs: cmap::launch_shape) TMA -> remainder -> MMA pipeline that runs across items.  The tensor core adds into its accumulator with
// truncation, so a long accumulation chain loses accuracy (1.4e-5 after the 192 MMAs of 512 input channels): an item is cut
// into SEGMENTS of 4 K chunks, the a_hi b_hi products (16 MMAs per segment) and the two cross terms go to separate accumulators,
// and the workers add the segments up in registers (round to nearest).  The accumulator pair is double-buffered in TMEM, so
// draining a segment overlaps the MMAs of the next one.  Warp 0 = TMA producer, warp 1 = MMA issue, warps 2-9 workers.
// =====================================================================================================================
constexpr int kGM = cmap::kM, kGN = cmap::kN, kGK = 32;   // voxels x outputs per item, channels per K chunk
constexpr int kGSeg = 4;                              // K chunks per accumulation segment
constexpr uint32_t kGA = kGK * kGM * 4;              // x chunk: 4 atoms of (32 channels x 32 voxels) = 16 KiB
constexpr uint32_t kGB = kGN * kGK * 4;              // W chunk: 64 rows x 128 bytes = 8 KiB
constexpr uint32_t gA = 0, gAlo = kGA, gB = 2 * kGA, gBlo = 2 * kGA + kGB, kGStage = 2 * kGA + 2 * kGB;   // 48 KiB
// barriers behind the stages: full / remainder-ready / empty per stage, accumulator full / free per accumulator pair, the TMEM slot
__host__ __device__ constexpr uint32_t g_smem_bytes(int stages) { return stages * kGStage + 3 * 8 * stages + 16 + 16 + 8; }

// x as (batch, channels, voxels): box (1, 32, 32), the 128-byte rows swizzled in 32-byte atoms
int make_map_x(CUtensorMap* m, const float* ptr, long long batch, int channels, long long voxels) {
    cuuint64_t dims[3] = {(cuuint64_t)voxels, (cuuint64_t)channels, (cuuint64_t)batch};
    cuuint64_t strides[2] = {(cuuint64_t)voxels * 4, (cuuint64_t)voxels * channels * 4};
    cuuint32_t box[3] = {32, kGK, 1};
    return encode_tiled_map(m, "x", CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, ptr, dims, strides, box,
                            CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
}
// W as (outputs, inputs) row-major: box (64 outputs, 32 inputs)
int make_map_w(CUtensorMap* m, const float* ptr, int cout, int cin) {
    cuuint64_t dims[2] = {(cuuint64_t)cin, (cuuint64_t)cout};
    cuuint64_t strides[1] = {(cuuint64_t)cin * 4};
    cuuint32_t box[2] = {kGK, kGN};
    return encode_tiled_map(m, "W", CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, ptr, dims, strides, box,
                            CU_TENSOR_MAP_SWIZZLE_128B);
}
// W stored as (inputs, outputs) row-major, used transposed (the input gradient reads the layer's weight as it lies): the
// outputs are contiguous, i.e. the B operand is MN-major like x: boxes of (32 outputs x 32 inputs), 128-byte rows swizzled in
// 32-byte atoms
int make_map_wt(CUtensorMap* m, const float* ptr, int cout, int cin) {
    cuuint64_t dims[2] = {(cuuint64_t)cout, (cuuint64_t)cin};
    cuuint64_t strides[1] = {(cuuint64_t)cout * 4};
    cuuint32_t box[2] = {32, kGK};
    return encode_tiled_map(m, "W^T", CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, ptr, dims, strides, box,
                            CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
}

// STAGES = 2: two CTAs per SM; STAGES = 4: one CTA per SM with four K chunks in flight (cmap::launch_shape)
template <int STAGES>
__global__ void __launch_bounds__(cmap::kThreads, STAGES <= 2 ? 2 : 1)
linear_fwd_tc(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w, const float* __restrict__ bias,
              float* __restrict__ y, const float* __restrict__ aux, float* __restrict__ y2, int epi, int wt, int cout, int cin, long long vox,
              int vtiles_per_sample, int otiles, long long total_items) {
    constexpr int kGStages = STAGES;
    constexpr uint32_t gBarFull = kGStages * kGStage, gBarLo = gBarFull + 8 * kGStages, gBarEmpty = gBarLo + 8 * kGStages,
                       gBarAccFull = gBarEmpty + 8 * kGStages, gBarAccFree = gBarAccFull + 16, gTmemSlot = gBarAccFree + 16;
    static_assert(gTmemSlot + 8 == g_smem_bytes(STAGES), "shared-memory map");
    extern __shared__ __align__(1024) unsigned char smem[];
    const uint32_t sbase = smem_u32(smem);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = (int)uniform_u32((uint32_t)(tid >> 5));
    const long long my_items = blockIdx.x < total_items ? (total_items - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int kchunks = (cin + kGK - 1) / kGK;

    if (tid == 0) {
        for (int s = 0; s < kGStages; ++s) {
            mbar_init(sbase + gBarFull + 8 * s, 1);
            mbar_init(sbase + gBarLo + 8 * s, 8);
            mbar_init(sbase + gBarEmpty + 8 * s, 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(sbase + gBarAccFull + 8 * a, 1);
            mbar_init(sbase + gBarAccFree + 8 * a, 8);
        }
        fence_mbarrier_init();
    }
    if (warp == 1) {
        tmem_alloc<256>(sbase + gTmemSlot);
        tmem_relinquish_alloc_permit();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = uniform_u32(*reinterpret_cast<const uint32_t*>(smem + gTmemSlot));

    if (warp == 0) {
        // ---- TMA producer: items in the order (voxel tile, output tile): neighbouring CTAs share the x tile in L2 ----
        if (elect_one()) {
            long long g = 0;
            for (long long it = 0; it < my_items; ++it) {
                const long long item = blockIdx.x + it * gridDim.x;
                const int ot = (int)(item % otiles);
                const long long vt_all = item / otiles;
                const int b = (int)(vt_all / vtiles_per_sample);
                const int v0 = (int)(vt_all - (long long)b * vtiles_per_sample) * kGM;
                for (int kc = 0; kc < kchunks; ++kc, ++g) {
                    const int s = (int)(g % kGStages);
                    const uint32_t round = (uint32_t)(g / kGStages);
                    if (round > 0) mbar_wait(sbase + gBarEmpty + 8 * s, (round - 1) & 1);
                    const uint32_t full = sbase + gBarFull + 8 * s, st = sbase + s * kGStage;
                    mbar_arrive_expect_tx(full, kGA + kGB);
#pragma unroll
                    for (int a = 0; a < 4; ++a) tma_load_3d(st + gA + a * (kGA / 4), &map_x, full, v0 + 32 * a, kc * kGK, b);
                    if (wt) {
                        tma_load_2d(st + gB, &map_w, full, ot * kGN, kc * kGK);
                        tma_load_2d(st + gB + kGB / 2, &map_w, full, ot * kGN + 32, kc * kGK);
                    } else {
                        tma_load_2d(st + gB, &map_w, full, kc * kGK, ot * kGN);
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ---- MMA issue ----
        const uint32_t idesc = make_idesc(128, kGN, true, wt != 0);        // A MN-major; B K-major, or MN-major for W^T
        const uint32_t b_lbo = wt ? kGB / 2 : 16, b_sbo = wt ? 512 : 1024, b_type = wt ? 1 : 2, b_kstep = wt ? 1024 : 32;
        long long g = 0, seg = 0;
        for (long long it = 0; it < my_items; ++it) {
            for (int kc = 0; kc < kchunks; ++kc, ++g) {
                const int ks = kc % kGSeg;                                 // position inside the segment
                const uint32_t acc = (uint32_t)(seg & 1), use = (uint32_t)(seg >> 1);
                if (ks == 0) {
                    if (use > 0) mbar_wait(sbase + gBarAccFree + 8 * acc, (use - 1) & 1);      // the workers have drained this pair
                    tc_fence_after();
                }
                const int s = (int)(g % kGStages);
                const uint32_t round = (uint32_t)(g / kGStages);
                mbar_wait(sbase + gBarLo + 8 * s, round & 1);
                tc_fence_after();
                const bool seg_end = ks + 1 == kGSeg || kc + 1 == kchunks;
                if (elect_one()) {
                    const uint32_t st = sbase + s * kGStage;
                    const uint64_t a_hi = make_desc(st + gA, kGA / 4, 512, 1), a_lo = make_desc(st + gAlo, kGA / 4, 512, 1);
                    const uint64_t b_hi = make_desc(st + gB, b_lbo, b_sbo, b_type), b_lo = make_desc(st + gBlo, b_lbo, b_sbo, b_type);
                    const uint32_t d_main = tmem + acc * (2 * kGN), d_cross = d_main + kGN;
#pragma unroll
                    for (int k = 0; k < kGK / 8; ++k) {
                        mma_tf32(d_cross, desc_at(a_lo, k * 1024), desc_at(b_hi, k * b_kstep), idesc, ks > 0 || k > 0);
                        mma_tf32(d_cross, desc_at(a_hi, k * 1024), desc_at(b_lo, k * b_kstep), idesc, 1);
                        mma_tf32(d_main, desc_at(a_hi, k * 1024), desc_at(b_hi, k * b_kstep), idesc, ks > 0 || k > 0);
                    }
                    commit(sbase + gBarEmpty + 8 * s);
                    if (seg_end) commit(sbase + gBarAccFull + 8 * acc);
                }
                __syncwarp();
                if (seg_end) ++seg;
            }
        }
    } else {
        // ---- workers: remainder tiles of every K chunk; a finished segment is drained after the first chunk of the next one ----
        const int t = tid - 64;                                            // 0 .. 255
        const int wq = warp & 3, wh = (warp - 2) >> 2;                     // TMEM lane quarter this warp may read; half of the columns
        const int spi = (kchunks + kGSeg - 1) / kGSeg;                     // segments per item
        float sum[32];
        const cmap::Epilogue<float> ep{bias, y, aux, y2, epi, cout, otiles, vtiles_per_sample, vox, wq, wh, lane};
        // an item's running sums are loaded an item ahead of their first use and cost no registers
        auto start_item = [&](long long it) {
#pragma unroll
            for (int i = 0; i < 32; ++i) sum[i] = 0.f;
            if (it < my_items) ep.start(sum, it, true);
        };
        start_item(0);
        auto drain = [&](long long seg) {
            const uint32_t acc = (uint32_t)(seg & 1), use = (uint32_t)(seg >> 1);
            mbar_wait(sbase + gBarAccFull + 8 * acc, use & 1);
            tc_fence_after();
            const uint32_t ta = tmem + ((uint32_t)(wq * 32) << 16) + acc * (2 * kGN) + wh * 32;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                uint32_t dm[16], dc[16];
                tmem_ld16_nowait(ta + h * 16, dm);
                tmem_ld16_nowait(ta + kGN + h * 16, dc);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 16; ++i) sum[h * 16 + i] += __uint_as_float(dm[i]) + __uint_as_float(dc[i]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(sbase + gBarAccFree + 8 * acc);
            if (seg % spi == spi - 1) {                                    // the item's last segment: epilogue, store, start over
                const long long it = seg / spi;
                ep.finish(sum, it);
                start_item(it + 1);
            }
        };
        long long g = 0, seg = 0;                                          // seg: the segment the current chunk belongs to
        for (long long it = 0; it < my_items; ++it) {
            for (int kc = 0; kc < kchunks; ++kc, ++g) {
                const int s = (int)(g % kGStages);
                const uint32_t round = (uint32_t)(g / kGStages);
                mbar_wait(sbase + gBarFull + 8 * s, round & 1);
                unsigned char* st = smem + s * kGStage;
                {
                    const float4* hi = reinterpret_cast<const float4*>(st + gA);
                    float4* lo = reinterpret_cast<float4*>(st + gAlo);
#pragma unroll
                    for (int i = 0; i < (int)(kGA / 16) / 256; ++i) {
                        const float4 v4 = hi[i * 256 + t];
                        lo[i * 256 + t] = make_float4(tf32_lo(v4.x), tf32_lo(v4.y), tf32_lo(v4.z), tf32_lo(v4.w));
                    }
                }
                {
                    const float4* hi = reinterpret_cast<const float4*>(st + gB);
                    float4* lo = reinterpret_cast<float4*>(st + gBlo);
#pragma unroll
                    for (int i = 0; i < (int)(kGB / 16) / 256; ++i) {
                        const float4 v4 = hi[i * 256 + t];
                        lo[i * 256 + t] = make_float4(tf32_lo(v4.x), tf32_lo(v4.y), tf32_lo(v4.z), tf32_lo(v4.w));
                    }
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(sbase + gBarLo + 8 * s);
                if (kc % kGSeg == 0 && seg > 0) drain(seg - 1);            // the previous segment, now that this one is under way
                if (kc % kGSeg == kGSeg - 1 || kc + 1 == kchunks) ++seg;
            }
        }
        if (seg > 0) drain(seg - 1);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<256>(tmem);
}

}  // namespace

bool linear_wgrad_tc_supported(const float* dy, const float* x, long long batch, int cout, int cin, long long voxels) {
    return voxels % 4 == 0 && voxels < (1LL << 31) && batch < (1LL << 31) && ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(x)) & 15) == 0 &&
           cout > 0 && cin > 0;
}

// dW / db must be zeroed by the caller (the kernel adds its CTA totals with atomics)
int linear_wgrad_tc_launch(const float* dy, const float* x, float* dW, float* db, long long batch, int cout, int cin, long long voxels,
                           cudaStream_t st) {
    CUtensorMap map_dy, map_x;
    if (int e = make_map(&map_dy, dy, batch, cout, voxels)) return e;
    if (int e = make_map(&map_x, x, batch, cin, voxels)) return e;
    static SmemConfig cfg;
    FZ_CUDA_CHECK(cfg.ensure(linear_wgrad_tc, kSmemW));
    const int tps = (int)((voxels + kVT - 1) / kVT);
    const long long tiles = batch * tps;
    const int bo = (cout + kBlk - 1) / kBlk, bi = (cin + kBlk - 1) / kBlk;
    const long long gx = cmap::wgrad_ctas((2LL * num_sms() + bo * bi - 1) / (bo * bi), tiles);
    linear_wgrad_tc<<<dim3((unsigned)gx, bo, bi), kThreads, kSmemW, st>>>(map_dy, map_x, dW, db, cout, cin, tps, tiles);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

}  // namespace fz

namespace fz {
bool linear_fwd_tc_supported(const float* x, const float* W, long long batch, int cout, int cin, long long voxels) {
    return voxels % 4 == 0 && cin % 4 == 0 && voxels < (1LL << 31) && batch < (1LL << 31) && cout > 0 && cin > 0 &&
           ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(W)) & 15) == 0;
}

int linear_fwd_tc_launch(const float* x, const float* W, const float* bias, float* y, const float* aux, float* y2, int epi,
                         int wt, long long batch, int cout, int cin, long long voxels, cudaStream_t st) {
    CUtensorMap map_x, map_w;
    if (int e = make_map_x(&map_x, x, batch, cin, voxels)) return e;
    if (int e = wt ? make_map_wt(&map_w, W, cout, cin) : make_map_w(&map_w, W, cout, cin)) return e;
    const int vtps = (int)((voxels + kGM - 1) / kGM);
    const int otiles = (cout + kGN - 1) / kGN;
    const long long items = batch * vtps * otiles;
    if (items >= (1LL << 31)) return fail(FZ_ERR_UNSUPPORTED, "linear forward: more than 2^31 (voxel tile, output tile) items");
    const cmap::Launch ls = cmap::launch_shape(items, (cin + kGK - 1) / kGK);
    if (ls.stages == 4) {
        static SmemConfig cfg4;
        FZ_CUDA_CHECK(cfg4.ensure(linear_fwd_tc<4>, g_smem_bytes(4)));
        linear_fwd_tc<4><<<ls.blocks, cmap::kThreads, g_smem_bytes(4), st>>>(map_x, map_w, bias, y, aux, y2, epi, wt, cout, cin, voxels, vtps,
                                                                            otiles, items);
    } else {
        static SmemConfig cfg2;
        FZ_CUDA_CHECK(cfg2.ensure(linear_fwd_tc<2>, g_smem_bytes(2)));
        linear_fwd_tc<2><<<ls.blocks, cmap::kThreads, g_smem_bytes(2), st>>>(map_x, map_w, bias, y, aux, y2, epi, wt, cout, cin, voxels, vtps,
                                                                            otiles, items);
    }
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}
}  // namespace fz
