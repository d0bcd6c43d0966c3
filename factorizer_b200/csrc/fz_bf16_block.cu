// The bf16 and fp16 FactorizerBlocks' channel maps on the tensor cores (tcgen05 kind::f16: bf16 or fp16 operands, fp32
// accumulator in TMEM), and the launch that stages their weights in 16 bits.  The U-Net scaffold's bf16 layers use the same
// channel maps and staging, and the stem's weight gradient below.  The kernels are templated on the 16-bit element type E,
// which sets the TMA data type, the MMA's operand format and the conversions (Elem16 below); nothing else differs.
//
// Channel map  y[b][o][v] = sum_c W[o][c] x[b][c][v] (+ bias[o]), with the item walk, the 2/4-stage launch policy and the five
// FZ_EPILOGUE_* epilogues it shares with linear_fwd_tc (fz_channel_map.cuh) -- one MMA per 16 channels and no remainder tiles:
//   D[128 voxels x 64 outputs] += A[128 x 64 channels] B[64 x 64]^T per K chunk (four MMAs),
// A = x, voxel-contiguous = MN-major: two TMA boxes of (64 channels x 64 voxels), each channel one 128-byte row in the
// 128-byte swizzle; B = W, K-major, one box of (64 outputs x 64 channels).  The weight is always K-major: the input
// gradient reads the transposed copy fz_bf16_stage_weights writes.  Bias, residual, GELU and GELU' are applied to the fp32
// sums, which are rounded to bf16 once.  The accumulator of an item is double-buffered in TMEM, so draining one item overlaps
// the MMAs of the next.  One chain per item: 512 channels are 32 MMAs, whose truncation (about 2^-24 S per MMA) stays far
// below the final bf16 rounding.  Warp 0 = TMA producer, warp 1 = MMA issue, warps 2-9 = epilogue (thread = voxel = TMEM lane,
// 32 outputs each).
//
// Weight gradient  dW[o][c] = sum over (batch, voxel) of dy[o][v] x[c][v], db[o] = sum of dy[o][v]: as linear_wgrad_tc,
// with bf16 K-major boxes of (128 channels x 64 voxels) and no remainder tiles: A = dy (M = 128 outputs), B = [x ; ones]
// (N = 128 inputs + the bias column), four MMAs per stage; dW, db fp32 with one atomic per element and CTA; the chain is
// capped at 32 stages per CTA as there (cmap::wgrad_ctas).
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "fz_channel_map.cuh"
#include "fz_internal.cuh"
#include "fz_tc.cuh"

namespace fz {
namespace {

using namespace tc;
typedef __nv_bfloat16 bf16;

template <typename E> struct Elem16;
template <> struct Elem16<bf16> {
    static constexpr CUtensorMapDataType kTma = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    static constexpr uint32_t kFormat = 1;             // instruction descriptor, A / B format
    static constexpr const char* kName = "bf16";
    static __device__ __forceinline__ bf16 from(float v) { return __float2bfloat16_rn(v); }
};
template <> struct Elem16<__half> {
    static constexpr CUtensorMapDataType kTma = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    static constexpr uint32_t kFormat = 0;
    static constexpr const char* kName = "fp16";
    static __device__ __forceinline__ __half from(float v) { return __float2half_rn(v); }
};

// ---- channel map ------------------------------------------------------------------------------------------------------------
constexpr int kHM = cmap::kM, kHN = cmap::kN, kHK = 64;   // voxels x outputs per item, channels per K chunk (one 128-byte row)
constexpr uint32_t kHA = kHK * kHM * 2;               // x chunk: two boxes of (64 channels x 64 voxels) = 16 KiB
constexpr uint32_t kHB = kHN * kHK * 2;               // W chunk: 64 rows x 128 bytes = 8 KiB
constexpr uint32_t hA = 0, hB = kHA, kHStage = kHA + kHB;
// barriers behind the stages: full / empty per stage, accumulator full / free per accumulator, the TMEM slot
__host__ __device__ constexpr uint32_t h_smem_bytes(int stages) { return stages * kHStage + 2 * 8 * stages + 16 + 16 + 8; }

// x as (batch, channels, voxels) of E: box (1, 64, 64)
template <typename E>
int make_map_x16(CUtensorMap* m, const E* ptr, long long batch, int channels, long long voxels) {
    cuuint64_t dims[3] = {(cuuint64_t)voxels, (cuuint64_t)channels, (cuuint64_t)batch};
    cuuint64_t strides[2] = {(cuuint64_t)voxels * 2, (cuuint64_t)voxels * channels * 2};
    cuuint32_t box[3] = {64, kHK, 1};
    return encode_tiled_map(m, "x (16-bit)", Elem16<E>::kTma, 3, ptr, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}
// a K-major matrix of E (rows, cols) with rows `ld` elements apart: box (box_rows, 64 columns)
// (rank 2, or rank 3 with `batch` such matrices rows * ld elements apart)
template <typename E>
int make_map_rows16(CUtensorMap* m, const char* what, const E* ptr, long long rows, long long cols, long long ld, int box_rows,
                    int rank, long long batch = 1) {
    cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)batch};
    cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)ld * rows * 2};
    cuuint32_t box[3] = {64, (cuuint32_t)box_rows, 1};
    return encode_tiled_map(m, what, Elem16<E>::kTma, rank, ptr, dims, strides, box,
                            CU_TENSOR_MAP_SWIZZLE_128B);
}

template <typename E, int STAGES>
__global__ void __launch_bounds__(cmap::kThreads, STAGES <= 2 ? 2 : 1)
linear_fwd_bf16_tc(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w, const float* __restrict__ bias,
                   E* __restrict__ y, const E* __restrict__ aux, E* __restrict__ y2, int epi, int cout, int cin, long long vox,
                   int vtiles_per_sample, int otiles, long long total_items) {
    constexpr uint32_t hBarFull = STAGES * kHStage, hBarEmpty = hBarFull + 8 * STAGES, hBarAccFull = hBarEmpty + 8 * STAGES,
                       hBarAccFree = hBarAccFull + 16, hTmemSlot = hBarAccFree + 16;
    static_assert(hTmemSlot + 8 == h_smem_bytes(STAGES), "shared-memory map");
    extern __shared__ __align__(1024) unsigned char smem[];
    const uint32_t sbase = smem_u32(smem);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = (int)uniform_u32((uint32_t)(tid >> 5));
    const long long my_items = blockIdx.x < total_items ? (total_items - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int kchunks = (cin + kHK - 1) / kHK;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(sbase + hBarFull + 8 * s, 1);
            mbar_init(sbase + hBarEmpty + 8 * s, 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(sbase + hBarAccFull + 8 * a, 1);
            mbar_init(sbase + hBarAccFree + 8 * a, 8);
        }
        fence_mbarrier_init();
    }
    if (warp == 1) {
        tmem_alloc<128>(sbase + hTmemSlot);
        tmem_relinquish_alloc_permit();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = uniform_u32(*reinterpret_cast<const uint32_t*>(smem + hTmemSlot));

    if (warp == 0) {
        // ---- TMA producer: items in the order (voxel tile, output tile): neighbouring CTAs share the x tile in L2 ----
        if (elect_one()) {
            long long g = 0;
            for (long long it = 0; it < my_items; ++it) {
                const long long item = blockIdx.x + it * gridDim.x;
                const int ot = (int)(item % otiles);
                const long long vt_all = item / otiles;
                const int b = (int)(vt_all / vtiles_per_sample);
                const int v0 = (int)(vt_all - (long long)b * vtiles_per_sample) * kHM;
                for (int kc = 0; kc < kchunks; ++kc, ++g) {
                    const int s = (int)(g % STAGES);
                    const uint32_t round = (uint32_t)(g / STAGES);
                    if (round > 0) mbar_wait(sbase + hBarEmpty + 8 * s, (round - 1) & 1);
                    const uint32_t full = sbase + hBarFull + 8 * s, st = sbase + s * kHStage;
                    mbar_arrive_expect_tx(full, kHA + kHB);
                    tma_load_3d(st + hA, &map_x, full, v0, kc * kHK, b);
                    tma_load_3d(st + hA + kHA / 2, &map_x, full, v0 + 64, kc * kHK, b);
                    tma_load_2d(st + hB, &map_w, full, kc * kHK, ot * kHN);
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ---- MMA issue: one accumulator per item, two in TMEM ----
        const uint32_t idesc = make_idesc_16bit(kHM, kHN, true, false, Elem16<E>::kFormat);   // A MN-major, B K-major
        long long g = 0;
        for (long long it = 0; it < my_items; ++it) {
            const uint32_t acc = (uint32_t)(it & 1), use = (uint32_t)(it >> 1);
            if (use > 0) mbar_wait(sbase + hBarAccFree + 8 * acc, (use - 1) & 1);   // the workers have drained this accumulator
            tc_fence_after();
            for (int kc = 0; kc < kchunks; ++kc, ++g) {
                const int s = (int)(g % STAGES);
                const uint32_t round = (uint32_t)(g / STAGES);
                mbar_wait(sbase + hBarFull + 8 * s, round & 1);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t st = sbase + s * kHStage;
                    const uint64_t ad = make_desc(st + hA, kHA / 2, 1024, 2), bd = make_desc(st + hB, 16, 1024, 2);
                    const uint32_t d = tmem + acc * kHN;
#pragma unroll
                    for (int k = 0; k < kHK / 16; ++k) mma_bf16(d, desc_at(ad, k * 2048), desc_at(bd, k * 32), idesc, kc > 0 || k > 0);
                    commit(sbase + hBarEmpty + 8 * s);
                    if (kc + 1 == kchunks) commit(sbase + hBarAccFull + 8 * acc);
                }
                __syncwarp();
            }
        }
    } else {
        // ---- workers: drain an item's accumulator, apply the epilogue in fp32, store E ----
        const int wq = warp & 3, wh = (warp - 2) >> 2;                     // TMEM lane quarter this warp may read; half of the columns
        const cmap::Epilogue<E> ep{bias, y, aux, y2, epi, cout, otiles, vtiles_per_sample, vox, wq, wh, lane};
        for (long long it = 0; it < my_items; ++it) {
            // the running sums start from the residual or the bias; their loads are in flight while the MMAs finish
            float sum[32];
#pragma unroll
            for (int o = 0; o < 32; ++o) sum[o] = 0.f;
            ep.start(sum, it, false);
            const uint32_t acc = (uint32_t)(it & 1), use = (uint32_t)(it >> 1);
            mbar_wait(sbase + hBarAccFull + 8 * acc, use & 1);
            tc_fence_after();
            const uint32_t ta = tmem + ((uint32_t)(wq * 32) << 16) + acc * kHN + wh * 32;
            uint32_t d0[16], d1[16];
            tmem_ld16_nowait(ta, d0);
            tmem_ld16_nowait(ta + 16, d1);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(sbase + hBarAccFree + 8 * acc);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                sum[i] += __uint_as_float(d0[i]);
                sum[16 + i] += __uint_as_float(d1[i]);
            }
            ep.finish(sum, it);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<128>(tmem);
}

// ---- weight gradient --------------------------------------------------------------------------------------------------------
constexpr int kWBlk = 128;                              // channels per block of dW, both ways
constexpr int kWVT = 64;                                // voxels per stage = one 128-byte swizzle row
constexpr int kWStages = 3;
constexpr int kWThreads = 192;
constexpr uint32_t kWTile = kWBlk * 128;                // one (128 x 64) 16-bit tile: 16 KiB
// stage: dy | x | ones block (16 rows: the first all ones)
constexpr uint32_t wA = 0, wB = kWTile, wOnes = 2 * kWTile, kWStage = 2 * kWTile + 16 * 128;
constexpr uint32_t wBarFull = kWStages * kWStage, wBarEmpty = wBarFull + 8 * kWStages, wBarDone = wBarEmpty + 8 * kWStages,
                   wTmemSlot = wBarDone + 8, kWSmem = wTmemSlot + 8;
constexpr int kWN = kWBlk + 16;                         // 144 accumulator columns
static_assert(kWBlk * (kWBlk + 17) * 4 <= kWStages * kWStage, "the epilogue's scratch copy fits in the stages");

template <typename E>
__global__ void __launch_bounds__(kWThreads, 2)
linear_wgrad_bf16_tc(const __grid_constant__ CUtensorMap map_dy, const __grid_constant__ CUtensorMap map_x, float* __restrict__ dW,
                     float* __restrict__ db, int cout, int cin, int tiles_per_sample, long long total_tiles) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const uint32_t sbase = smem_u32(smem);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = (int)uniform_u32((uint32_t)(tid >> 5));
    const int ob = blockIdx.y, ib = blockIdx.z;
    const long long my_tiles = blockIdx.x < total_tiles ? (total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (tid == 0) {
        for (int s = 0; s < kWStages; ++s) {
            mbar_init(sbase + wBarFull + 8 * s, 1);
            mbar_init(sbase + wBarEmpty + 8 * s, 1);
        }
        mbar_init(sbase + wBarDone, 1);
        fence_mbarrier_init();
    }
    // the ones block of every stage (constant): row 0 = ones, rows 1 .. 15 = zeros (a 128-byte row of equal values: no swizzle to mind)
    for (int i = tid; i < kWStages * 16 * 64; i += kWThreads) {
        const int s = i / (16 * 64), r = (i / 64) % 16;
        reinterpret_cast<E*>(smem + s * kWStage + wOnes)[i % (16 * 64)] = Elem16<E>::from(r == 0 ? 1.f : 0.f);
    }
    if (warp == 1) {
        tmem_alloc<256>(sbase + wTmemSlot);
        tmem_relinquish_alloc_permit();
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = uniform_u32(*reinterpret_cast<const uint32_t*>(smem + wTmemSlot));

    if (warp == 0) {
        // ---- TMA producer ----
        if (elect_one()) {
            long long nb = (long long)blockIdx.x / tiles_per_sample;
            int nt = (int)((long long)blockIdx.x - nb * tiles_per_sample);
            for (long long it = 0; it < my_tiles; ++it) {
                const int s = (int)(it % kWStages);
                const uint32_t round = (uint32_t)(it / kWStages);
                if (round > 0) mbar_wait(sbase + wBarEmpty + 8 * s, (round - 1) & 1);
                const uint32_t full = sbase + wBarFull + 8 * s;
                mbar_arrive_expect_tx(full, 2 * kWTile);
                tma_load_3d(sbase + s * kWStage + wA, &map_dy, full, nt * kWVT, ob * kWBlk, (int)nb);
                tma_load_3d(sbase + s * kWStage + wB, &map_x, full, nt * kWVT, ib * kWBlk, (int)nb);
                nt += (int)gridDim.x;
                while (nt >= tiles_per_sample) { nt -= tiles_per_sample; ++nb; }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ---- MMA issue: D[128 x 144] += dy (rows) x [x ; ones] (columns) over the stage's 4 groups of 16 voxels ----
        const uint32_t idesc = make_idesc_16bit(kWBlk, kWN, false, false, Elem16<E>::kFormat);
        for (long long it = 0; it < my_tiles; ++it) {
            const int s = (int)(it % kWStages);
            const uint32_t round = (uint32_t)(it / kWStages);
            mbar_wait(sbase + wBarFull + 8 * s, round & 1);
            tc_fence_after();
            if (elect_one()) {
                const uint64_t ad = make_desc(sbase + s * kWStage + wA, 16, 1024, 2);
                const uint64_t bd = make_desc(sbase + s * kWStage + wB, 16, 1024, 2);
#pragma unroll
                for (int k = 0; k < kWVT / 16; ++k) mma_bf16(tmem, desc_at(ad, k * 32), desc_at(bd, k * 32), idesc, it > 0 || k > 0);
                commit(sbase + wBarEmpty + 8 * s);
                if (it + 1 == my_tiles) commit(sbase + wBarDone);
            }
            __syncwarp();
        }
    }
    // ---- epilogue: accumulator row r (TMEM lane r) = output channel r; column n < 128 = input channel n, column 128 = the bias sums ----
    if (my_tiles > 0) {
        mbar_wait(sbase + wBarDone, 0);
        tc_fence_after();
    }
    __syncthreads();                                           // the stages are free: they take the scratch copy of the accumulator
    float* S = reinterpret_cast<float*>(smem);                 // [128][145]
    constexpr int kS = kWBlk + 17;
    if (my_tiles > 0 && warp >= 2) {
        const int q = warp & 3;                                // the TMEM lane quarter this warp may read
        const int r = q * 32 + lane;
        const uint32_t row_addr = tmem + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
        for (int c0 = 0; c0 < kWBlk; c0 += 32) {
            float d[32];
            tmem_ld32(row_addr + c0, d);
#pragma unroll
            for (int c = 0; c < 32; ++c) S[r * kS + c0 + c] = d[c];
        }
        uint32_t e[16];
        tmem_ld16_nowait(row_addr + kWBlk, e);
        tmem_ld_wait();
        S[r * kS + kWBlk] = __uint_as_float(e[0]);
    }
    tc_fence_before();
    __syncthreads();
    if (my_tiles > 0) {
        for (int i = tid; i < kWBlk * kWBlk; i += kWThreads) {
            const int o = i / kWBlk, c = i % kWBlk;
            const int go = ob * kWBlk + o, gc = ib * kWBlk + c;
            if (go < cout && gc < cin) atomicAdd(dW + (size_t)go * cin + gc, S[o * kS + c]);
        }
        if (db && ib == 0 && tid < kWBlk && ob * kWBlk + tid < cout) atomicAdd(db + ob * kWBlk + tid, S[tid * kS + kWBlk]);
    }
    __syncthreads();
    if (warp == 1) tmem_dealloc<256>(tmem);
}

// ---- stem weight gradient ---------------------------------------------------------------------------------------------------
// dW[o][r] = sum over voxels of dy[o][v] col[r][v], with col[r = (c, kd, kh, kw)][v] = x[c][v + (kd-1, kh-1, kw-1)] (zero
// outside the volume): the 27 cin im2col rows of a 64-voxel tile are built in shared memory, never in global memory, in the
// K-major SWIZZLE_128B layout TMA writes (row r = 128 bytes, its 16-byte chunk j at (j ^ (r % 8))); row 27 cin is all ones (its
// sums are db), the rest zero.  D[128 rows x 32 outputs] += col[128 x 64] dy[32 x 64]^T, four MMAs per stage; dy comes by TMA.
// Warp 0 = TMA, warp 1 = MMA issue, warps 2-9 = im2col builders, then the epilogue (one atomic per element and CTA).  The chain
// is capped at 32 stages per CTA, as in linear_wgrad_bf16_tc.
constexpr int kSV = 64;                                 // voxels per stage
constexpr int kSStages = 3;
constexpr int kSThreads = 320;
constexpr int kSBuilders = kSThreads - 64;
constexpr uint32_t kSA = 128 * 128, kSB = 32 * 128, kSStage = kSA + kSB;     // im2col tile 16 KiB | dy tile 4 KiB
constexpr uint32_t sBarFull = kSStages * kSStage, sBarEmpty = sBarFull + 8 * kSStages, sBarDone = sBarEmpty + 8 * kSStages,
                   sTmemSlot = sBarDone + 8, kSSmem = sTmemSlot + 8;

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}

template <typename TX>
__global__ void __launch_bounds__(kSThreads, 1)
stem_wgrad_bf16_tc(const __grid_constant__ CUtensorMap map_dy, const TX* __restrict__ x, float* __restrict__ dW, float* __restrict__ db,
                   int cin, int D, int H, int W, int tiles_per_sample, long long total_tiles) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const uint32_t sbase = smem_u32(smem);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = (int)uniform_u32((uint32_t)(tid >> 5));
    const int R = 27 * cin;
    const long long vox = (long long)D * H * W;
    const long long my_tiles = blockIdx.x < total_tiles ? (total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (tid == 0) {
        for (int s = 0; s < kSStages; ++s) {
            mbar_init(sbase + sBarFull + 8 * s, 1 + kSBuilders / 32);
            mbar_init(sbase + sBarEmpty + 8 * s, 1);
        }
        mbar_init(sbase + sBarDone, 1);
        fence_mbarrier_init();
    }
    // the constant rows of every stage: R = ones, R+1 .. 127 = zeros (rows of equal values: no swizzle to mind)
    for (int i = tid; i < kSStages * (128 - R) * 64; i += kSThreads) {
        const int s = i / ((128 - R) * 64), e = i % ((128 - R) * 64);
        reinterpret_cast<bf16*>(smem + s * kSStage)[R * 64 + e] = __float2bfloat16_rn(e < 64 ? 1.f : 0.f);
    }
    if (warp == 1) {
        tmem_alloc<32>(sbase + sTmemSlot);
        tmem_relinquish_alloc_permit();
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = uniform_u32(*reinterpret_cast<const uint32_t*>(smem + sTmemSlot));

    if (warp == 0) {
        // ---- TMA producer: the dy tile (32 outputs x 64 voxels) ----
        if (elect_one()) {
            for (long long it = 0; it < my_tiles; ++it) {
                const long long tile = blockIdx.x + it * gridDim.x;
                const int nb = (int)(tile / tiles_per_sample), nt = (int)(tile - (long long)nb * tiles_per_sample);
                const int s = (int)(it % kSStages);
                const uint32_t round = (uint32_t)(it / kSStages);
                if (round > 0) mbar_wait(sbase + sBarEmpty + 8 * s, (round - 1) & 1);
                const uint32_t full = sbase + sBarFull + 8 * s;
                mbar_arrive_expect_tx(full, kSB);
                tma_load_3d(sbase + s * kSStage + kSA, &map_dy, full, nt * kSV, 0, nb);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ---- MMA issue ----
        const uint32_t idesc = make_idesc_bf16(128, 32, false, false);
        for (long long it = 0; it < my_tiles; ++it) {
            const int s = (int)(it % kSStages);
            const uint32_t round = (uint32_t)(it / kSStages);
            mbar_wait(sbase + sBarFull + 8 * s, round & 1);
            tc_fence_after();
            if (elect_one()) {
                const uint64_t ad = make_desc(sbase + s * kSStage, 16, 1024, 2);
                const uint64_t bd = make_desc(sbase + s * kSStage + kSA, 16, 1024, 2);
#pragma unroll
                for (int k = 0; k < kSV / 16; ++k) mma_bf16(tmem, desc_at(ad, k * 32), desc_at(bd, k * 32), idesc, it > 0 || k > 0);
                commit(sbase + sBarEmpty + 8 * s);
                if (it + 1 == my_tiles) commit(sbase + sBarDone);
            }
            __syncwarp();
        }
    } else {
        // ---- im2col builders: a thread fills 16-byte chunks (8 voxels along W, W % 8 == 0) of rows r, r + 32, ... ----
        const int b = tid - 64, j = b & 7, r0 = b >> 3;
        for (long long it = 0; it < my_tiles; ++it) {
            const long long tile = blockIdx.x + it * gridDim.x;
            const long long nb = tile / tiles_per_sample;
            const long long v = (tile - nb * tiles_per_sample) * kSV + 8 * j;
            const int w = (int)(v % W), h = (int)((v / W) % H), d = (int)(v / ((long long)W * H));
            const bool live = v < vox;
            const TX* xb = x + nb * cin * vox;
            const int s = (int)(it % kSStages);
            const uint32_t round = (uint32_t)(it / kSStages);
            if (round > 0) mbar_wait(sbase + sBarEmpty + 8 * s, (round - 1) & 1);
            unsigned char* tileA = smem + s * kSStage;
            for (int r = r0; r < R; r += kSBuilders / 8) {
                const int c = r / 27, t = r - 27 * c, kd = t / 9, kh = (t / 3) % 3, kw = t % 3;
                const int dd = d + kd - 1, hh = h + kh - 1, w0 = w + kw - 1;
                const bool rowok = live && dd >= 0 && dd < D && hh >= 0 && hh < H;
                const TX* src = xb + c * vox + ((long long)dd * H + hh) * W + w0;
                float e[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) e[i] = (rowok && w0 + i >= 0 && w0 + i < W) ? cmap::ldg_f(src + i) : 0.f;
                const uint4 q = make_uint4(pack_bf16(e[0], e[1]), pack_bf16(e[2], e[3]), pack_bf16(e[4], e[5]), pack_bf16(e[6], e[7]));
                *reinterpret_cast<uint4*>(tileA + r * 128 + ((j ^ (r & 7)) << 4)) = q;
            }
            fence_proxy_async_smem();                          // generic-proxy writes -> the tensor core's reads
            __syncwarp();
            if (lane == 0) mbar_arrive(sbase + sBarFull + 8 * s);
        }
    }
    // ---- epilogue: TMEM lane r = im2col row r, column o = output channel ----
    if (warp >= 2 && my_tiles > 0) {
        mbar_wait(sbase + sBarDone, 0);
        tc_fence_after();
        const int q = warp & 3, half = (warp - 2) >> 2;       // TMEM lane quarter; columns [16 half, 16 half + 16)
        const int r = q * 32 + lane;
        uint32_t e[16];
        tmem_ld16_nowait(tmem + ((uint32_t)(q * 32) << 16) + 16 * half, e);
        tmem_ld_wait();
        if (r < R) {
#pragma unroll
            for (int i = 0; i < 16; ++i) atomicAdd(dW + (16 * half + i) * R + r, __uint_as_float(e[i]));
        } else if (r == R && db) {
#pragma unroll
            for (int i = 0; i < 16; ++i) atomicAdd(db + 16 * half + i, __uint_as_float(e[i]));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<32>(tmem);
}

// ---- weight staging ---------------------------------------------------------------------------------------------------------
// 16-bit rows are padded to whole 16-byte groups: a TMA row stride must be a multiple of 16 bytes
__host__ __device__ inline long long ld8(long long n) { return (n + 7) & ~7LL; }

struct StageArgs {
    const float* w[4];
    int rows[4], cols[4];
    long long off[9];                                           // start of each of the 8 outputs (W_i, W_i^T), and the total
};

template <typename E>
__global__ void __launch_bounds__(256) stage_weights_bf16(StageArgs a, E* __restrict__ out) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.off[8]; i += (long long)gridDim.x * blockDim.x) {
        int j = 0;
#pragma unroll
        for (int q = 1; q < 8; ++q) j += i >= a.off[q];
        const int m = j >> 1;
        const int R = a.rows[m], C = a.cols[m];
        const long long local = i - a.off[j];
        float v = 0.f;
        if ((j & 1) == 0) {                                      // W (R, C) as stored, rows ld8(C) apart
            const long long ld = ld8(C), r = local / ld, c = local - r * ld;
            if (c < C) v = __ldg(a.w[m] + r * C + c);
        } else {                                                 // W^T (C, R), rows ld8(R) apart
            const long long ld = ld8(R), c = local / ld, r = local - c * ld;
            if (r < R) v = __ldg(a.w[m] + r * C + c);
        }
        out[i] = Elem16<E>::from(v);
    }
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

template <typename E>
int stage_weights_launch(int n, const float* const* w, const int* r, const int* c, void* out, void* stream) {
    tls().launches = 0;
    StageArgs a;
    long long off = 0;
    for (int m = 0; m < 4; ++m) {
        if (m >= n) {                                           // absent weights: empty ranges at the end
            a.w[m] = nullptr;
            a.rows[m] = a.cols[m] = 1;
            a.off[2 * m] = a.off[2 * m + 1] = off;
            continue;
        }
        if (!w[m] || !fz_bf16_stage_weights_supported(r[m], c[m])) return fail(FZ_ERR_INVALID, "weight %d: null or bad shape (%d, %d)", m, r[m], c[m]);
        a.w[m] = w[m];
        a.rows[m] = r[m];
        a.cols[m] = c[m];
        a.off[2 * m] = off;
        off += (long long)r[m] * ld8(c[m]);
        a.off[2 * m + 1] = off;
        off += (long long)c[m] * ld8(r[m]);
    }
    a.off[8] = off;
    if (!out) return fail(FZ_ERR_INVALID, "null buffer");
    if (!aligned16(out)) return fail(FZ_ERR_UNSUPPORTED, "staged weights must be 16-byte aligned");
    long long blocks = (off + 255) / 256;
    if (blocks > 4LL * num_sms()) blocks = 4LL * num_sms();
    stage_weights_bf16<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a, static_cast<E*>(out));
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

bool channel_map16_supported(int32_t cout, int32_t cin, int64_t voxels) {
    return cout > 0 && cin > 0 && voxels > 0 && voxels % 8 == 0 && voxels < (1LL << 31);
}

template <typename E>
int linear_forward16(const void* x, const void* W, int32_t ldw, const float* bias, void* y, int64_t batch, int32_t cin, int32_t cout,
                     int64_t voxels, int32_t epilogue, const void* aux, void* y2, void* stream) {
    const char* nm = Elem16<E>::kName;
    tls().launches = 0;
    if (batch == 0) return FZ_OK;
    if (!x || !W || !y) return fail(FZ_ERR_INVALID, "null buffer");
    if (batch < 0 || batch >= (1LL << 31)) return fail(FZ_ERR_INVALID, "batch=%lld", (long long)batch);
    char what[32];
    snprintf(what, sizeof(what), "%s channel map", nm);
    if (int e = cmap::check_epilogue(what, epilogue, aux, y2)) return e;
    if (!channel_map16_supported(cout, cin, voxels))
        return fail(FZ_ERR_UNSUPPORTED, "%s channel map: voxels must be a positive multiple of 8 below 2^31 (got %lld)", nm, (long long)voxels);
    if (ldw < cin || ldw % 8) return fail(FZ_ERR_UNSUPPORTED, "%s channel map: ldw=%d must be >= cin=%d and a multiple of 8", nm, ldw, cin);
    if (!aligned16(x) || !aligned16(W))
        return fail(FZ_ERR_UNSUPPORTED, "%s channel map: x and W must be 16-byte aligned", nm);
    if (((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(aux) | reinterpret_cast<uintptr_t>(y2)) & 1))
        return fail(FZ_ERR_UNSUPPORTED, "%s channel map: y, aux and y2 must be 2-byte aligned", nm);
    CUtensorMap map_x, map_w;
    if (int e = make_map_x16(&map_x, static_cast<const E*>(x), batch, cin, voxels)) return e;
    if (int e = make_map_rows16(&map_w, "W (16-bit)", static_cast<const E*>(W), cout, cin, ldw, kHN, 2)) return e;
    const int vtps = (int)((voxels + kHM - 1) / kHM);
    const int otiles = (cout + kHN - 1) / kHN;
    const long long items = batch * vtps * otiles;
    if (items >= (1LL << 31)) return fail(FZ_ERR_UNSUPPORTED, "%s channel map: more than 2^31 (voxel tile, output tile) items", nm);
    E* ye = static_cast<E*>(y);
    E* y2e = static_cast<E*>(y2);
    const E* ae = static_cast<const E*>(aux);
    cudaStream_t st = (cudaStream_t)stream;
    const cmap::Launch ls = cmap::launch_shape(items, (cin + kHK - 1) / kHK);
    if (ls.stages == 4) {
        static SmemConfig cfg4;
        FZ_CUDA_CHECK(cfg4.ensure(linear_fwd_bf16_tc<E, 4>, h_smem_bytes(4)));
        linear_fwd_bf16_tc<E, 4><<<ls.blocks, cmap::kThreads, h_smem_bytes(4), st>>>(map_x, map_w, bias, ye, ae, y2e, epilogue, cout, cin,
                                                                                    voxels, vtps, otiles, items);
    } else {
        static SmemConfig cfg2;
        FZ_CUDA_CHECK(cfg2.ensure(linear_fwd_bf16_tc<E, 2>, h_smem_bytes(2)));
        linear_fwd_bf16_tc<E, 2><<<ls.blocks, cmap::kThreads, h_smem_bytes(2), st>>>(map_x, map_w, bias, ye, ae, y2e, epilogue, cout, cin,
                                                                                    voxels, vtps, otiles, items);
    }
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

template <typename E>
int linear_wgrad16(const void* dy, const void* x, float* dW, float* db, int64_t batch, int32_t cout, int32_t cin, int64_t voxels,
                   void* stream) {
    const char* nm = Elem16<E>::kName;
    tls().launches = 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (!dW) return fail(FZ_ERR_INVALID, "null buffer");
    if (cout < 1 || cin < 1 || batch < 0 || batch >= (1LL << 31)) return fail(FZ_ERR_INVALID, "bad sizes");
    FZ_CUDA_CHECK(cudaMemsetAsync(dW, 0, sizeof(float) * (size_t)cout * cin, st));
    if (db) FZ_CUDA_CHECK(cudaMemsetAsync(db, 0, sizeof(float) * (size_t)cout, st));
    if (batch == 0 || voxels == 0) return FZ_OK;
    if (!dy || !x) return fail(FZ_ERR_INVALID, "null buffer");
    if (!channel_map16_supported(cout, cin, voxels))
        return fail(FZ_ERR_UNSUPPORTED, "%s weight gradient: voxels must be a positive multiple of 8 below 2^31 (got %lld)", nm, (long long)voxels);
    if (!aligned16(dy) || !aligned16(x)) return fail(FZ_ERR_UNSUPPORTED, "%s weight gradient: dy and x must be 16-byte aligned", nm);
    CUtensorMap map_dy, map_x;
    if (int e = make_map_rows16(&map_dy, "dy (16-bit)", static_cast<const E*>(dy), cout, voxels, voxels, kWBlk, 3, batch)) return e;
    if (int e = make_map_rows16(&map_x, "x (16-bit)", static_cast<const E*>(x), cin, voxels, voxels, kWBlk, 3, batch)) return e;
    static SmemConfig cfg;
    FZ_CUDA_CHECK(cfg.ensure(linear_wgrad_bf16_tc<E>, kWSmem));
    const int tps = (int)((voxels + kWVT - 1) / kWVT);
    const long long tiles = batch * tps;
    const int bo = (cout + kWBlk - 1) / kWBlk, bi = (cin + kWBlk - 1) / kWBlk;
    const long long gx = cmap::wgrad_ctas((2LL * num_sms() + bo * bi - 1) / (bo * bi), tiles);
    linear_wgrad_bf16_tc<E><<<dim3((unsigned)gx, bo, bi), kWThreads, kWSmem, st>>>(map_dy, map_x, dW, db, cout, cin, tps, tiles);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

}  // namespace
}  // namespace fz

using namespace fz;

extern "C" {

int fz_linear_forward_bf16_supported(int32_t cout, int32_t cin, int64_t voxels) { return channel_map16_supported(cout, cin, voxels); }

int fz_linear_forward_bf16(const void* x, const void* W, int32_t ldw, const float* bias, void* y, int64_t batch, int32_t cin, int32_t cout,
                           int64_t voxels, int32_t epilogue, const void* aux, void* y2, void* stream) {
    return linear_forward16<bf16>(x, W, ldw, bias, y, batch, cin, cout, voxels, epilogue, aux, y2, stream);
}

int fz_linear_wgrad_bf16_supported(int32_t cout, int32_t cin, int64_t voxels) { return channel_map16_supported(cout, cin, voxels); }

int fz_linear_wgrad_bf16(const void* dy, const void* x, float* dW, float* db, int64_t batch, int32_t cout, int32_t cin, int64_t voxels,
                         void* stream) {
    return linear_wgrad16<bf16>(dy, x, dW, db, batch, cout, cin, voxels, stream);
}

int fz_bf16_stage_weights_supported(int32_t rows, int32_t cols) {
    return rows > 0 && cols > 0 && (long long)ld8(rows) * ld8(cols) < (1LL << 28);
}

int64_t fz_bf16_staged_elems(int32_t rows, int32_t cols) {
    return (int64_t)rows * ld8(cols) + (int64_t)cols * ld8(rows);
}

int fz_bf16_stage_weights(const float* w0, int32_t r0, int32_t c0, const float* w1, int32_t r1, int32_t c1, const float* w2, int32_t r2,
                          int32_t c2, const float* w3, int32_t r3, int32_t c3, void* out, void* stream) {
    const float* w[4] = {w0, w1, w2, w3};
    const int r[4] = {r0, r1, r2, r3}, c[4] = {c0, c1, c2, c3};
    return stage_weights_launch<bf16>(4, w, r, c, out, stream);
}

int fz_bf16_stage_weight(const float* w, int32_t rows, int32_t cols, void* out, void* stream) {
    return stage_weights_launch<bf16>(1, &w, &rows, &cols, out, stream);
}

int fz_linear_forward_f16_supported(int32_t cout, int32_t cin, int64_t voxels) { return channel_map16_supported(cout, cin, voxels); }

int fz_linear_forward_f16(const void* x, const void* W, int32_t ldw, const float* bias, void* y, int64_t batch, int32_t cin, int32_t cout,
                          int64_t voxels, int32_t epilogue, const void* aux, void* y2, void* stream) {
    return linear_forward16<__half>(x, W, ldw, bias, y, batch, cin, cout, voxels, epilogue, aux, y2, stream);
}

int fz_linear_wgrad_f16_supported(int32_t cout, int32_t cin, int64_t voxels) { return channel_map16_supported(cout, cin, voxels); }

int fz_linear_wgrad_f16(const void* dy, const void* x, float* dW, float* db, int64_t batch, int32_t cout, int32_t cin, int64_t voxels,
                        void* stream) {
    return linear_wgrad16<__half>(dy, x, dW, db, batch, cout, cin, voxels, stream);
}

int fz_f16_stage_weights_supported(int32_t rows, int32_t cols) { return fz_bf16_stage_weights_supported(rows, cols); }

int64_t fz_f16_staged_elems(int32_t rows, int32_t cols) { return fz_bf16_staged_elems(rows, cols); }

int fz_f16_stage_weights(const float* w0, int32_t r0, int32_t c0, const float* w1, int32_t r1, int32_t c1, const float* w2, int32_t r2,
                         int32_t c2, const float* w3, int32_t r3, int32_t c3, void* out, void* stream) {
    const float* w[4] = {w0, w1, w2, w3};
    const int r[4] = {r0, r1, r2, r3}, c[4] = {c0, c1, c2, c3};
    return stage_weights_launch<__half>(4, w, r, c, out, stream);
}

int fz_f16_stage_weight(const float* w, int32_t rows, int32_t cols, void* out, void* stream) {
    return stage_weights_launch<__half>(1, &w, &rows, &cols, out, stream);
}

int fz_conv3d_stem_wgrad_bf16_supported(int32_t cin, int32_t cout, int32_t D, int32_t H, int32_t W) {
    return cin >= 1 && cin <= 4 && cout == 32 && D > 0 && H > 0 && W > 0 && W % 8 == 0 && (long long)D * H * W < (1LL << 31);
}

int fz_conv3d_stem_wgrad_bf16(const void* dy, const void* x, int32_t x_dtype, float* dW, float* db, int64_t batch, int32_t cin, int32_t cout,
                              int32_t D, int32_t H, int32_t W, void* stream) {
    tls().launches = 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (!dW) return fail(FZ_ERR_INVALID, "null buffer");
    if (batch < 0 || batch >= (1LL << 31)) return fail(FZ_ERR_INVALID, "stem weight gradient: bad batch");
    if (x_dtype != FZ_DTYPE_F32 && x_dtype != FZ_DTYPE_BF16) return fail(FZ_ERR_INVALID, "stem weight gradient: unknown x dtype %d", x_dtype);
    if (!fz_conv3d_stem_wgrad_bf16_supported(cin, cout, D, H, W))
        return fail(FZ_ERR_UNSUPPORTED, "stem weight gradient handles 1..4 -> 32 channels, W divisible by 8 (got %d -> %d, W = %d)", cin, cout, W);
    FZ_CUDA_CHECK(cudaMemsetAsync(dW, 0, sizeof(float) * (size_t)cout * cin * 27, st));
    if (db) FZ_CUDA_CHECK(cudaMemsetAsync(db, 0, sizeof(float) * (size_t)cout, st));
    if (batch == 0) return FZ_OK;
    if (!dy || !x) return fail(FZ_ERR_INVALID, "null buffer");
    if (!aligned16(dy) || !aligned16(x)) return fail(FZ_ERR_UNSUPPORTED, "stem weight gradient: dy and x must be 16-byte aligned");
    const long long vox = (long long)D * H * W;
    CUtensorMap map_dy;
    if (int e = make_map_rows16(&map_dy, "dy (bf16)", static_cast<const bf16*>(dy), cout, vox, vox, 32, 3, batch)) return e;
    const int tps = (int)((vox + kSV - 1) / kSV);
    const long long tiles = batch * tps;
    const long long gx = cmap::wgrad_ctas(2LL * num_sms(), tiles);
    if (gx >= (1LL << 31)) return fail(FZ_ERR_UNSUPPORTED, "stem weight gradient: too many voxels");
    if (x_dtype == FZ_DTYPE_F32) {
        static SmemConfig cfg;
        FZ_CUDA_CHECK(cfg.ensure(stem_wgrad_bf16_tc<float>, kSSmem));
        stem_wgrad_bf16_tc<float><<<(unsigned)gx, kSThreads, kSSmem, st>>>(map_dy, static_cast<const float*>(x), dW, db, cin, D, H, W, tps, tiles);
    } else {
        static SmemConfig cfg;
        FZ_CUDA_CHECK(cfg.ensure(stem_wgrad_bf16_tc<bf16>, kSSmem));
        stem_wgrad_bf16_tc<bf16><<<(unsigned)gx, kSThreads, kSSmem, st>>>(map_dy, static_cast<const bf16*>(x), dW, db, cin, D, H, W, tps, tiles);
    }
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

}  // extern "C"
