// Three-launch scheme of the "octant" formulation of the fused FactMixer core (see fz_swnmf_octant.cuh for the
// formulation and the per-tile / per-window device code): pass 1, pass 2 and pass 3 are separate launches over the
// whole volume.  Used for volumes that fit the L2 anyway (nothing to gain from pipelining the passes), as the inner
// step of the paired-window-set variant at the end of this file, and as the reference the pipelined scheme
// (fz_swnmf_pipe.cu, the production path for large volumes) is tested against.
#include <initializer_list>
#include <type_traits>

#include "fz_swnmf_octant.cuh"

namespace fz {
using namespace oct;
namespace {

constexpr int kW1 = 7;                // warps per CTA, pass 1 forward (2 x 16 KiB each)
constexpr int kW3 = 6;                // pass 3 forward (2 x 16 KiB each; 7 warps measured slower: 111 vs 97 us)
constexpr int kWB = 3;                // passes 1 and 3 backward (2 x 32 KiB each)
constexpr int kSolveThreads = 64;      // backward pass 2: a lane per window, small CTAs so that 64 Ki windows spread over all SMs

// one streaming warp: its tiles are gw, gw + nw, ...; buffers are filled one tile ahead by lane 0
struct Stream {
    int gw, nw, lane;
    int begin, count, reverse;       // this launch covers tiles [begin, begin + count), possibly walked backwards
    __device__ __forceinline__ int tile(int k) const {
        const int i = gw + k * nw;
        if (i >= count) return 0x7fffffff;
        return begin + (reverse ? count - 1 - i : i);
    }
};

// The kernels are templated on the volume's element type E: float, or 16-bit activations (__nv_bfloat16, __half).  With 16-bit
// activations a streaming warp's unit of work is a PAIR of tiles side by side along W, fetched as one (16,8,8,8) box of 16-bit
// values = the same 16 KiB and the same 32-byte rows as one fp32 tile; the pair is then worked on as two tiles, and whatever
// is prefetched for "the next tile" (window factors) is prefetched per tile of the pair.
// Stream::tile(k) counts units: tiles (fp32) or pairs (16-bit); a pair is tiles 2u and 2u + 1 (t2 is the fastest index).
template <typename E> constexpr int kPerUnit = std::is_same<E, float>::value ? 1 : 2;    // tiles per unit
template <typename E> struct TileOf { typedef Tile16<E> type; };
template <> struct TileOf<float> { typedef TileF32 type; };
template <typename E>
__device__ __forceinline__ typename TileOf<E>::type tile_at(const float* buf, int half) {
    if constexpr (kPerUnit<E> == 2) return Tile16<E>{reinterpret_cast<const unsigned char*>(buf) + 16 * half};
    else return TileF32{buf};
}

// =====================================================================================================
// forward pass 1: per-octant Gram partials of every unshifted tile
// =====================================================================================================
template <typename E>
__global__ void __launch_bounds__(kW1 * 32, 1) phase_fwd_gram(const __grid_constant__ PhaseParams P) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(16) float v0s[512];
    __shared__ uint64_t bars[kW1][2];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* buf = reinterpret_cast<float*>(smem_raw) + (size_t)warp * 2 * 4096;
    for (int j = threadIdx.x; j < 512; j += blockDim.x) v0s[j] = P.v0[j];
    if (lane == 0) {
        mbar_init(&bars[warp][0], 1);
        mbar_init(&bars[warp][1], 1);
        fence_mbarrier_init();
    }
    __syncthreads();
    if (blockIdx.x == 0 && warp == 0) {
        // b_1 = v_0 . v_0 is the same for every window: computed once, here
        float sq = 0.f;
        for (int j = lane; j < 512; j += 32) sq = fmaf(v0s[j], v0s[j], sq);
        sq = warp_sum_f(sq);
        if (lane == 0) *P.b1 = sq;
    }
    constexpr int kPer = kPerUnit<E>;
    const int units = P.t_count / kPer;
    Stream S; S.gw = blockIdx.x * kW1 + warp; S.nw = gridDim.x * kW1; S.lane = lane; S.begin = P.t_begin / kPer; S.count = units; S.reverse = 0;
    int dst[15];
    gram_destinations(lane, dst);
    auto issue = [&](int k) {
        const int u = S.tile(k);
        if (u < P.tiles && lane == 0) {
            const TileCoord c = tile_coord(P, u * kPer);
            mbar_arrive_expect_tx(&bars[warp][k & 1], kTileBytes);
            tma_load_tile(buf + (k & 1) * 4096, &P.tm_x, &bars[warp][k & 1], c.t2 * 8, c.t1 * 8, c.t0 * 8, c.h * 8, c.b);
        }
    };
    issue(0);
    uint32_t parity[2] = {0, 0};
    for (int k = 0; S.tile(k) < P.tiles; ++k) {
        __syncwarp();            // everyone is done with the buffer that is refilled now
        issue(k + 1);
        const int u = S.tile(k), st = k & 1;
        mbar_wait(&bars[warp][st], parity[st]);
        parity[st] ^= 1;
        if constexpr (kPer == 2) {
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
                // the record is assembled in the pair buffer's first 16-byte column: tile 0 of the pair is in registers
                // by then (half 0) or long consumed (half 1)
                fwd_tile_gram<Tile16<E>, 2>(tile_at<E>(buf + st * 4096, half), buf + st * 4096, v0s, dst, lane,
                                           P.oct + (size_t)(2 * u + half) * kTileRec);
                __syncwarp();
            }
        } else {
            fwd_tile_gram(buf + st * 4096, v0s, dst, lane, P.oct + (size_t)u * kTileRec);
        }
    }
}

// =====================================================================================================
// forward pass 2: per window (either set), 8 lanes: add the 8 octant records, run the T sweeps
// =====================================================================================================
__global__ void __launch_bounds__(128) phase_fwd_solve(const __grid_constant__ PhaseParams P) {
    // 8 lanes per window.  (A lane-per-window variant, 5x fewer instructions, measured SLOWER here: 27 us against 18 us --
    // its 2 048 warps each walk 8 dependent rounds of record loads; the backward's recursion is long enough to gain.)
    __shared__ __align__(16) float sums[128 / 8][64];               // per window: Gam (36) | r (8) | a1 set 0 | a1 set 1
    const int lane = threadIdx.x & 31, grp = threadIdx.x >> 3;
    long long gidx = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
    const bool active = gidx < 2LL * P.t_count;     // a group past the end computes window 0 along with its warp, stores nothing
    if (!active) gidx = 0;
    const int set = gidx >= P.t_count ? 1 : 0;
    const long long gwin = (long long)set * P.tiles + P.t_begin + (gidx - (long long)set * P.t_count);
    fwd_solve_window(P, &sums[grp][0], gwin, set, lane, active, __ldcg(P.b1));
}

// =====================================================================================================
// forward pass 3: y = 1/2 (u_0 v_0^T + u_1 v_1^T) voxel by voxel, v_s = relu(rd_s (X^T u_s + eps))
// OutT: the volume's own type, or fp32 for a 16-bit volume whose y is a partial sum (the paired window sets below)
// =====================================================================================================
template <typename E, typename OutT = E>
__global__ void __launch_bounds__(kW3 * 32, 1) phase_fwd_apply(const __grid_constant__ PhaseParams P) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ uint64_t bars[kW3][2];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* buf = reinterpret_cast<float*>(smem_raw) + (size_t)warp * 2 * 4096;
    if (lane == 0) {
        mbar_init(&bars[warp][0], 1);
        mbar_init(&bars[warp][1], 1);
        fence_mbarrier_init();
    }
    __syncthreads();
    constexpr int kPer = kPerUnit<E>;
    Stream S; S.gw = blockIdx.x * kW3 + warp; S.nw = gridDim.x * kW3; S.lane = lane; S.begin = P.t_begin / kPer; S.count = P.t_count / kPer; S.reverse = P.reverse;
    const int oct = lane >> 2;

    auto issue = [&](int k) {
        const int u = S.tile(k);
        if (u < P.tiles && lane == 0) {
            const TileCoord c = tile_coord(P, u * kPer);
            mbar_arrive_expect_tx(&bars[warp][k & 1], kTileBytes);
            tma_load_tile(buf + (k & 1) * 4096, &P.tm_x, &bars[warp][k & 1], c.t2 * 8, c.t1 * 8, c.t0 * 8, c.h * 8, c.b);
        }
    };
    // tile number q of this warp's sequence of TILES (fp32: unit q; 16-bit: tile q % 2 of unit q / 2)
    auto tile_of = [&](int q) -> int {
        const int u = S.tile(q / kPer);
        return u < P.tiles ? u * kPer + (q % kPer) : 0x7fffffff;
    };
    auto factors = [&](int q, Fac& f0, Fac& f1) {
        const int tid = tile_of(q);
        if (tid < P.tiles) {
            const TileCoord c = tile_coord(P, tid);
            f0 = load_fac(P.fac, tid);
            f1 = load_fac(P.fac, (long long)P.tiles + shifted_window_of(P, c, oct));
        }
    };
    issue(0);
    Fac n0, n1;
    factors(0, n0, n1);
    uint32_t parity[2] = {0, 0};
    for (int k = 0; S.tile(k) < P.tiles; ++k) {
        __syncwarp();
        issue(k + 1);
        const int st = k & 1;
#pragma unroll 1
        for (int half = 0; half < kPer; ++half) {
            const int q = k * kPer + half;
            const Fac f0 = n0, f1 = n1;
            factors(q + 1, n0, n1);
            const TileCoord c = tile_coord(P, tile_of(q));
            if (half == 0) {
                mbar_wait(&bars[warp][st], parity[st]);
                parity[st] ^= 1;
            }
            fwd_tile_apply_t<kPer == 1, false, typename TileOf<E>::type, OutT>(P, tile_at<E>(buf + st * 4096, half), f0, f1, c, lane);
        }
    }
}

// =====================================================================================================
// backward pass 1: per octant and window set, lane-partials of  w = G v_T / 2 + X cbar_T  and  e = qbar_T . v_T
// =====================================================================================================
template <typename E>
__global__ void __launch_bounds__(kWB * 32, 1) phase_bwd_reduce(const __grid_constant__ PhaseParams P) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ uint64_t bars[kWB][2];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* buf = reinterpret_cast<float*>(smem_raw) + (size_t)warp * 4 * 4096;    // [stage][X | G]
    if (lane == 0) {
        mbar_init(&bars[warp][0], 1);
        mbar_init(&bars[warp][1], 1);
        fence_mbarrier_init();
    }
    __syncthreads();
    constexpr int kPer = kPerUnit<E>;
    Stream S; S.gw = blockIdx.x * kWB + warp; S.nw = gridDim.x * kWB; S.lane = lane; S.begin = P.t_begin / kPer; S.count = P.t_count / kPer; S.reverse = 0;
    const int oct = lane >> 2;

    auto issue = [&](int k) {
        const int u = S.tile(k);
        if (u < P.tiles && lane == 0) {
            const TileCoord c = tile_coord(P, u * kPer);
            float* b = buf + (k & 1) * 8192;
            mbar_arrive_expect_tx(&bars[warp][k & 1], 2 * kTileBytes);
            tma_load_tile(b, &P.tm_x, &bars[warp][k & 1], c.t2 * 8, c.t1 * 8, c.t0 * 8, c.h * 8, c.b);
            tma_load_tile(b + 4096, &P.tm_g, &bars[warp][k & 1], c.t2 * 8, c.t1 * 8, c.t0 * 8, c.h * 8, c.b);
        }
    };
    auto tile_of = [&](int q) -> int {
        const int u = S.tile(q / kPer);
        return u < P.tiles ? u * kPer + (q % kPer) : 0x7fffffff;
    };
    auto factors = [&](int q, UT& f0, UT& f1) {
        const int tid = tile_of(q);
        if (tid < P.tiles) {
            const TileCoord c = tile_coord(P, tid);
            f0 = load_ut(P, tid);
            f1 = load_ut(P, (long long)P.tiles + shifted_window_of(P, c, oct));
        }
    };
    issue(0);
    UT n0, n1;
    factors(0, n0, n1);
    uint32_t parity[2] = {0, 0};
    for (int k = 0; S.tile(k) < P.tiles; ++k) {
        __syncwarp();
        issue(k + 1);
        const int st = k & 1;
#pragma unroll 1
        for (int half = 0; half < kPer; ++half) {
            const int q = k * kPer + half;
            const UT f0 = n0, f1 = n1;
            factors(q + 1, n0, n1);
            const int tid = tile_of(q);
            if (half == 0) {
                mbar_wait(&bars[warp][st], parity[st]);
                parity[st] ^= 1;
            }
            bwd_tile_reduce_t(P, tile_at<E>(buf + st * 8192, half), tile_at<E>(buf + st * 8192 + 4096, half), f0, f1, lane,
                              P.oct + (size_t)tid * kBwdTileRec);
        }
    }
}

// =====================================================================================================
// backward pass 2: per window, 8 lanes: the 8-vector recursion t = T .. 1 (fz_swnmf_gram.cuh header)
// =====================================================================================================
__global__ void __launch_bounds__(kSolveThreads) phase_bwd_solve(const __grid_constant__ PhaseParams P) {
    long long gidx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = gidx < 2LL * P.t_count;
    if (!active) gidx = 0;
    const int set = gidx >= P.t_count ? 1 : 0;
    const long long gwin = (long long)set * P.tiles + P.t_begin + (gidx - (long long)set * P.t_count);
    bwd_solve_lane(P, gwin, set, active);
}

// =====================================================================================================
// backward pass 3: dx = [x > 0] sum_s ( rd_s u_s (u_s . g)/2 + M_s x + m_s + abar1_s v0[col_s] ) voxel by voxel
// OutT as in forward pass 3
// =====================================================================================================
template <typename E, typename OutT = E>
__global__ void __launch_bounds__(kWB * 32, 1) phase_bwd_apply(const __grid_constant__ PhaseParams P) {
    constexpr int kPer = kPerUnit<E>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(16) float v0s[512];
    __shared__ __align__(16) float mbs_all[kWB][2][9 * kMbF];     // [tile parity][window record: 0 = unshifted, 1 + o = shifted window of octant o]
    __shared__ uint64_t bars[kWB][2];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* buf = reinterpret_cast<float*>(smem_raw) + (size_t)warp * 4 * 4096;
    for (int j = threadIdx.x; j < 512; j += blockDim.x) v0s[j] = P.v0[j];
    if (lane == 0) {
        mbar_init(&bars[warp][0], 1);
        mbar_init(&bars[warp][1], 1);
        fence_mbarrier_init();
    }
    __syncthreads();
    Stream S; S.gw = blockIdx.x * kWB + warp; S.nw = gridDim.x * kWB; S.lane = lane; S.begin = P.t_begin / kPer; S.count = P.t_count / kPer; S.reverse = P.reverse;

    // the tile data of unit k (a tile, or a pair of 16-bit tiles): one TMA box each for X and dY
    auto issue = [&](int k) {
        const int u = S.tile(k);
        if (u < P.tiles && lane == 0) {
            const TileCoord c = tile_coord(P, u * kPer);
            uint64_t* bar = &bars[warp][k & 1];
            float* b = buf + (k & 1) * 8192;
            mbar_arrive_expect_tx(bar, 2 * kTileBytes);
            tma_load_tile(b, &P.tm_x, bar, c.t2 * 8, c.t1 * 8, c.t0 * 8, c.h * 8, c.b);
            tma_load_tile(b + 4096, &P.tm_g, bar, c.t2 * 8, c.t1 * 8, c.t0 * 8, c.h * 8, c.b);
        }
    };
    // tile number q of this warp's sequence of TILES (fp32: unit q; 16-bit: tile q % 2 of unit q / 2)
    auto tile_of = [&](int q) -> int {
        const int u = S.tile(q / kPer);
        return u < P.tiles ? u * kPer + (q % kPer) : 0x7fffffff;
    };
    // the nine window records of tile q, one tile ahead of the arithmetic: cp.async group q
    auto fetch = [&](int q) {
        const int tid = tile_of(q);
        if (tid < P.tiles) bwd_fetch_records(P, mbs_all[warp][q & 1], tid, tile_coord(P, tid), lane);
        cp_async_commit();
    };
    issue(0);
    fetch(0);
    uint32_t parity[2] = {0, 0};
    for (int k = 0; S.tile(k) < P.tiles; ++k) {
        __syncwarp();
        issue(k + 1);
        const int st = k & 1;
#pragma unroll 1
        for (int half = 0; half < kPer; ++half) {
            const int q = k * kPer + half;
            fetch(q + 1);
            cp_async_wait<1>();     // this lane's copies of tile q have landed ...
            __syncwarp();                                             // ... and so have everyone else's
            if (half == 0) {
                mbar_wait(&bars[warp][st], parity[st]);
                parity[st] ^= 1;
            }
            const TileCoord c = tile_coord(P, tile_of(q));
            bwd_tile_apply_t<false, typename TileOf<E>::type, OutT>(
                P, tile_at<E>(buf + st * 8192, half), tile_at<E>(buf + st * 8192 + 4096, half), mbs_all[warp][q & 1], v0s, c, lane);
            __syncwarp();                                             // records of tile q are free for tile q + 2
        }
    }
}

// ---- host ------------------------------------------------------------------------------------------------
struct Layout { size_t oct, b1, fac, mb, total; };
Layout layout(const DevGeom& G) {
    const size_t tiles = (size_t)G.mats_per_shift;
    Layout L;
    L.oct = 0;
    const size_t oct_bytes = tiles * kTileRec * sizeof(float);     // forward records (the backward's are smaller)
    L.b1 = align_up(oct_bytes, 256);
    L.fac = L.b1 + 256;
    L.mb = L.fac + align_up(2 * tiles * kFacF * sizeof(float), 256);
    L.total = L.mb + align_up(2 * tiles * kMbF * sizeof(float), 256);
    return L;
}

void fill(PhaseParams& P, const DevGeom& G, const fz_solver& s, int K, void* workspace) {
    fill_common(P, G, s, K);
    const Layout L = layout(G);
    char* ws = static_cast<char*>(workspace);
    P.oct = reinterpret_cast<float*>(ws + L.oct);
    P.b1 = reinterpret_cast<float*>(ws + L.b1);
    P.fac = reinterpret_cast<float*>(ws + L.fac);
    P.mb = reinterpret_cast<float*>(ws + L.mb);
}

int grid_for(int tiles, int warps) {
    int ctas = (tiles + warps - 1) / warps;
    return ctas < num_sms() ? ctas : num_sms();
}

// the three forward / backward passes over P's tiles for volumes of E; f32_out: y / dX are fp32 partial sums
template <typename E>
int forward_passes(const PhaseParams& P, bool f32_out, cudaStream_t st) {
    static SmemConfig cfg_gram, cfg_apply, cfg_apply_f;
    FZ_CUDA_CHECK(cfg_gram.ensure(phase_fwd_gram<E>, kW1 * 2 * kTileBytes));
    if (f32_out) FZ_CUDA_CHECK(cfg_apply_f.ensure(phase_fwd_apply<E, float>, kW3 * 2 * kTileBytes));
    else FZ_CUDA_CHECK(cfg_apply.ensure(phase_fwd_apply<E>, kW3 * 2 * kTileBytes));
    const int units = P.t_count / kPerUnit<E>;           // streaming warps work on tiles (fp32) or pairs of tiles (16-bit)
    phase_fwd_gram<E><<<grid_for(units, kW1), kW1 * 32, kW1 * 2 * kTileBytes, st>>>(P);
    FZ_LAUNCH_CHECK();
    const long long groups = 2LL * P.t_count;
    phase_fwd_solve<<<(unsigned)((groups * 8 + 127) / 128), 128, 0, st>>>(P);
    FZ_LAUNCH_CHECK();
    if (f32_out) phase_fwd_apply<E, float><<<grid_for(units, kW3), kW3 * 32, kW3 * 2 * kTileBytes, st>>>(P);
    else phase_fwd_apply<E><<<grid_for(units, kW3), kW3 * 32, kW3 * 2 * kTileBytes, st>>>(P);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

template <typename E>
int backward_passes(const PhaseParams& P, bool f32_out, cudaStream_t st) {
    static SmemConfig cfg_reduce, cfg_apply, cfg_apply_f;
    FZ_CUDA_CHECK(cfg_reduce.ensure(phase_bwd_reduce<E>, kWB * 4 * kTileBytes));
    if (f32_out) FZ_CUDA_CHECK(cfg_apply_f.ensure(phase_bwd_apply<E, float>, kWB * 4 * kTileBytes));
    else FZ_CUDA_CHECK(cfg_apply.ensure(phase_bwd_apply<E>, kWB * 4 * kTileBytes));
    const int units = P.t_count / kPerUnit<E>;
    phase_bwd_reduce<E><<<grid_for(units, kWB), kWB * 32, kWB * 4 * kTileBytes, st>>>(P);
    FZ_LAUNCH_CHECK();
    const long long groups = 2LL * P.t_count;
    phase_bwd_solve<<<(unsigned)((groups + kSolveThreads - 1) / kSolveThreads), kSolveThreads, 0, st>>>(P);
    FZ_LAUNCH_CHECK();
    if (f32_out) phase_bwd_apply<E, float><<<grid_for(units, kWB), kWB * 32, kWB * 4 * kTileBytes, st>>>(P);
    else phase_bwd_apply<E><<<grid_for(units, kWB), kWB * 32, kWB * 4 * kTileBytes, st>>>(P);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

}  // namespace

bool phase_supported(const DevGeom& G, const fz_solver& s, int relu) {
    if (!relu || s.kind != FZ_SOLVER_HALS || s.rank != 1) return false;
    if (s.num_iters < 1 || s.num_iters > 8) return false;
    if (G.d != 8 || G.p[0] != 8 || G.p[1] != 8 || G.p[2] != 8 || G.S != 2) return false;
    if (G.mats_per_shift == 0 || G.mats_per_shift >= (1LL << 28)) return false;
    if (G.dtype != FZ_DTYPE_F32 && (G.g[2] % 2)) return false;       // 16-bit tiles travel in pairs along W
    for (int k = 0; k < 3; ++k) {
        int a = G.sh[0][k] % G.n[k], b = G.sh[1][k] % G.n[k];
        if (a < 0) a += G.n[k];
        if (b < 0) b += G.n[k];
        if (a != 0 || b != 4) return false;
    }
    return true;
}

size_t phase_workspace_bytes(const DevGeom& G, const fz_solver& s) {
    (void)s;
    return layout(G).total;
}

int phase_forward(const float* x, const float* v0, float* y, void* saved, void* workspace,
                  const DevGeom& G, const fz_solver& s, cudaStream_t st, bool f32_out) {
    if (!workspace) return fail(FZ_ERR_INVALID, "fz_swnmf_forward: workspace of %zu bytes required", phase_workspace_bytes(G, s));
    if (reinterpret_cast<uintptr_t>(y) & 15) return fail(FZ_ERR_INVALID, "output pointer %p is not 16-byte aligned", (void*)y);
    static thread_local PhaseParams P;
    fill(P, G, s, 0, workspace);
    if (int e = make_tile_map(&P.tm_x, x, G)) return e;
    P.x = x; P.out = y; P.v0 = v0; P.saved = static_cast<float*>(saved);
    P.t_begin = 0;
    P.t_count = P.tiles;
    P.reverse = 1;          // pass 3 walks the tiles backwards: the tail of pass 1 is what L2 still holds
    if (G.dtype == FZ_DTYPE_BF16) return forward_passes<__nv_bfloat16>(P, f32_out, st);
    if (G.dtype == FZ_DTYPE_F16) return forward_passes<__half>(P, f32_out, st);
    return forward_passes<float>(P, false, st);
}

int phase_backward(const float* x, const float* gy, const float* v0, const void* saved, float* gx,
                   void* workspace, const DevGeom& G, const fz_solver& s, int K, cudaStream_t st, bool f32_out) {
    if (!workspace) return fail(FZ_ERR_INVALID, "fz_swnmf_backward: workspace of %zu bytes required", phase_workspace_bytes(G, s));
    if (!saved) return fail(FZ_ERR_INVALID, "fz_swnmf_backward: the `saved` buffer written by fz_swnmf_forward is required");
    if (reinterpret_cast<uintptr_t>(gx) & 15) return fail(FZ_ERR_INVALID, "output pointer %p is not 16-byte aligned", (void*)gx);
    static thread_local PhaseParams P;
    fill(P, G, s, K, workspace);
    if (int e = make_tile_map(&P.tm_x, x, G)) return e;
    if (int e = make_tile_map(&P.tm_g, gy, G)) return e;
    P.x = x; P.gy = gy; P.out = gx; P.v0 = v0;
    P.saved = const_cast<float*>(static_cast<const float*>(saved));
    P.t_begin = 0;
    P.t_count = P.tiles;
    P.reverse = 1;
    if (G.dtype == FZ_DTYPE_BF16) return backward_passes<__nv_bfloat16>(P, f32_out, st);
    if (G.dtype == FZ_DTYPE_F16) return backward_passes<__half>(P, f32_out, st);
    return backward_passes<float>(P, false, st);
}


// =====================================================================================================
// Window sets that pair up as (a, a + patch/2): every pair is the octant problem on the volume rolled by a
//   sum_{s in {a, a+4}} inv_s(NMF(win(roll(x, s)))) = roll( octant(roll(x, a)), -a )
// (torch.roll composes: roll(x, a + 4) = roll(roll(x, a), 4); operations.py:266-280), so e.g. the brats23
// bundle's shifts [0, 2, 4, 6] (model_zoo/factorizer_brats23/configs/train.yaml:50-54) run as two octant
// problems plus one roll and one roll-and-combine pass per pair instead of four window-at-a-time sweeps.  A bf16 or fp16
// volume is rolled in its own type (an exact 2-byte copy) and the pairs' partial sums stay fp32 until the last combine writes
// the 16-bit result.
// =====================================================================================================
namespace {

struct RollParams { int n0, n1, n2, s0, s1, s2; long long rows, vox; };

// V neighbouring elements as one access: fp32 8 or 16 bytes, bf16 / fp16 4 or 8 bytes
template <typename T, int V> struct VecOf { typedef typename std::conditional<V == 4, uint2, unsigned int>::type type; };
template <> struct VecOf<float, 2> { typedef float2 type; };
template <> struct VecOf<float, 4> { typedef float4 type; };

// two fp32 sums rounded once to a 16-bit pair
__device__ __forceinline__ void round_pair(__nv_bfloat162* p, float a, float b) { *p = __floats2bfloat162_rn(a, b); }
__device__ __forceinline__ void round_pair(__half2* p, float a, float b) { *p = __floats2half2_rn(a, b); }

// out[r][i] = in[r][(i - s) mod n]   (torch.roll), an exact copy for either element type.  One CTA per (row, i0) plane;
// V = 2 or 4 neighbouring voxels per thread (n2 and s2 multiples of V), 32-bit index math.
template <typename T, int V>
__global__ void __launch_bounds__(256) roll_volume(const T* __restrict__ in, T* __restrict__ out, const RollParams R) {
    typedef typename VecOf<T, V>::type vec;
    const int hv = R.n2 / V, per_plane = R.n1 * hv;
    for (long long pl = blockIdx.x; pl < R.rows * R.n0; pl += gridDim.x) {
        const long long r = pl / R.n0;
        const int i0 = (int)(pl - r * R.n0);
        int j0 = i0 - R.s0;
        if (j0 < 0) j0 += R.n0;
        const T* src = in + r * R.vox + (long long)j0 * R.n1 * R.n2;
        T* dst = out + r * R.vox + (long long)i0 * R.n1 * R.n2;
        for (int t = threadIdx.x; t < per_plane; t += blockDim.x) {
            const int i1 = t / hv, i2 = (t - i1 * hv) * V;
            int j1 = i1 - R.s1, j2 = i2 - R.s2;
            if (j1 < 0) j1 += R.n1;
            if (j2 < 0) j2 += R.n2;
            *reinterpret_cast<vec*>(dst + i1 * R.n2 + i2) = __ldcs(reinterpret_cast<const vec*>(src + j1 * R.n2 + j2));
        }
    }
}

// acc[r][i] = ((first ? 0 : acc[r][i]) + part[r][(i + s) mod n]) * scale   (the inverse roll, summed over the pairs).
// T = bf16 / fp16: the last call for a 16-bit volume, which writes that sum to y[r][i] instead of acc, rounded to T once
// (T = float leaves y unused).
template <int V, typename T>
__global__ void __launch_bounds__(256) unroll_combine(float* __restrict__ acc, const float* __restrict__ part, const RollParams R,
                                                      int first, float scale, T* __restrict__ y) {
    typedef typename std::conditional<V == 4, float4, float2>::type vec;
    const int hv = R.n2 / V, per_plane = R.n1 * hv;
    for (long long pl = blockIdx.x; pl < R.rows * R.n0; pl += gridDim.x) {
        const long long r = pl / R.n0;
        const int i0 = (int)(pl - r * R.n0);
        int j0 = i0 + R.s0;
        if (j0 >= R.n0) j0 -= R.n0;
        const float* src = part + r * R.vox + (long long)j0 * R.n1 * R.n2;
        float* dst = acc + r * R.vox + (long long)i0 * R.n1 * R.n2;
        for (int t = threadIdx.x; t < per_plane; t += blockDim.x) {
            const int i1 = t / hv, i2 = (t - i1 * hv) * V;
            int j1 = i1 + R.s1, j2 = i2 + R.s2;
            if (j1 >= R.n1) j1 -= R.n1;
            if (j2 >= R.n2) j2 -= R.n2;
            vec v = __ldcs(reinterpret_cast<const vec*>(src + j1 * R.n2 + j2));
            float* vf = reinterpret_cast<float*>(&v);
            vec* d = reinterpret_cast<vec*>(dst + i1 * R.n2 + i2);
            if (!first) {
                const vec o = *d;
                const float* of = reinterpret_cast<const float*>(&o);
#pragma unroll
                for (int q = 0; q < V; ++q) vf[q] += of[q];
            }
#pragma unroll
            for (int q = 0; q < V; ++q) vf[q] *= scale;
            if constexpr (std::is_same<T, float>::value) {
                *d = v;
            } else {
                typedef typename std::conditional<std::is_same<T, __half>::value, __half2, __nv_bfloat162>::type T2;
                typename VecOf<T, V>::type h;
                T2* hp = reinterpret_cast<T2*>(&h);
#pragma unroll
                for (int q = 0; q < V / 2; ++q) round_pair(hp + q, vf[2 * q], vf[2 * q + 1]);
                *reinterpret_cast<typename VecOf<T, V>::type*>(y + r * R.vox + (long long)i0 * R.n1 * R.n2 + i1 * R.n2 + i2) = h;
            }
        }
    }
}

int norm_shift(int v, int n) { v %= n; return v < 0 ? v + n : v; }

// base shift of every pair (normalised to [0, n)); false if the sets do not pair up
bool find_pairs(const DevGeom& G, int (*base)[3]) {
    if (G.S < 2 || G.S % 2) return false;
    bool used[FZ_MAX_SHIFTS] = {false};
    int np = 0;
    for (int a = 0; a < G.S; ++a) {
        if (used[a]) continue;
        int b = -1;
        for (int c = 0; c < G.S && b < 0; ++c) {
            if (c == a || used[c]) continue;
            bool ok = true;
            for (int k = 0; k < 3; ++k)
                if (norm_shift(G.sh[c][k] - G.sh[a][k], G.n[k]) != 4 % G.n[k]) ok = false;
            if (ok) b = c;
        }
        if (b < 0) return false;
        used[a] = used[b] = true;
        for (int k = 0; k < 3; ++k) base[np][k] = norm_shift(G.sh[a][k], G.n[k]);
        ++np;
    }
    return true;
}

DevGeom pair_geom(const DevGeom& G) {
    DevGeom P = G;
    P.S = 2;
    for (int q = 0; q < FZ_MAX_SHIFTS; ++q)
        for (int k = 0; k < 3; ++k) P.sh[q][k] = q == 1 ? 4 : 0;
    return P;
}

size_t vol_bytes(const DevGeom& G, size_t elem) { return align_up((size_t)G.B * G.C * G.vox * elem, 256); }
size_t elem_bytes(const DevGeom& G) { return G.dtype != FZ_DTYPE_F32 ? 2 : sizeof(float); }

// The workspace of the paired scheme: the octant kernels' own, then the rolled x and the rolled dY (the volume's element
// type), the partial sum of one pair (fp32) and, for 16-bit volumes, the fp32 sum over the pairs (fp32 volumes sum in y / dX).
struct PairBufs { float *xr, *gr, *part, *acc; };
PairBufs pair_bufs(void* workspace, const DevGeom& G, const fz_solver& s, float* out) {
    char* p = static_cast<char*>(workspace) + align_up(phase_workspace_bytes(pair_geom(G), s), 256);
    PairBufs b;
    b.xr = reinterpret_cast<float*>(p);
    p += vol_bytes(G, elem_bytes(G));
    b.gr = reinterpret_cast<float*>(p);
    p += vol_bytes(G, elem_bytes(G));
    b.part = reinterpret_cast<float*>(p);
    p += vol_bytes(G, sizeof(float));
    b.acc = G.dtype != FZ_DTYPE_F32 ? reinterpret_cast<float*>(p) : out;
    return b;
}

template <typename T>
void roll_as(const float* in, float* out, const RollParams& R, bool v4, unsigned grid, cudaStream_t st) {
    const T* i = reinterpret_cast<const T*>(in);
    T* o = reinterpret_cast<T*>(out);
    if (v4) roll_volume<T, 4><<<grid, 256, 0, st>>>(i, o, R);
    else roll_volume<T, 2><<<grid, 256, 0, st>>>(i, o, R);
}
int launch_roll(const float* in, float* out, const DevGeom& G, const int* a, cudaStream_t st) {
    RollParams R = {G.n[0], G.n[1], G.n[2], a[0], a[1], a[2], (long long)G.B * G.C, G.vox};
    const long long planes = R.rows * R.n0;
    const unsigned grid = (unsigned)(planes < 65535LL * 16 ? planes : 65535LL * 16);
    const bool v4 = R.n2 % 4 == 0 && R.s2 % 4 == 0;
    if (G.dtype == FZ_DTYPE_BF16) roll_as<__nv_bfloat16>(in, out, R, v4, grid, st);
    else if (G.dtype == FZ_DTYPE_F16) roll_as<__half>(in, out, R, v4, grid, st);
    else roll_as<float>(in, out, R, v4, grid, st);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}
template <typename T>
void combine_into(float* acc, const float* part, const RollParams& R, int first, float scale, float* y, bool v4, unsigned grid,
                  cudaStream_t st) {
    T* h = reinterpret_cast<T*>(y);
    if (v4) unroll_combine<4, T><<<grid, 256, 0, st>>>(acc, part, R, first, scale, h);
    else unroll_combine<2, T><<<grid, 256, 0, st>>>(acc, part, R, first, scale, h);
}
// adds pair partial `part` into acc; y: the last call for a 16-bit volume, which writes the finished sum there in its type
int launch_combine(float* acc, const float* part, const DevGeom& G, const int* a, int first, float scale, float* y, cudaStream_t st) {
    RollParams R = {G.n[0], G.n[1], G.n[2], a[0], a[1], a[2], (long long)G.B * G.C, G.vox};
    const long long planes = R.rows * R.n0;
    const unsigned grid = (unsigned)(planes < 65535LL * 16 ? planes : 65535LL * 16);
    const bool v4 = R.n2 % 4 == 0 && R.s2 % 4 == 0;
    if (y && G.dtype == FZ_DTYPE_F16) {
        combine_into<__half>(acc, part, R, first, scale, y, v4, grid, st);
    } else if (y) {
        combine_into<__nv_bfloat16>(acc, part, R, first, scale, y, v4, grid, st);
    } else {
        if (v4) unroll_combine<4, float><<<grid, 256, 0, st>>>(acc, part, R, first, scale, nullptr);
        else unroll_combine<2, float><<<grid, 256, 0, st>>>(acc, part, R, first, scale, nullptr);
    }
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

int check_16bit_pointers(std::initializer_list<const void*> ptrs) {
    for (const void* p : ptrs)
        if (reinterpret_cast<uintptr_t>(p) & 15) return fail(FZ_ERR_INVALID, "16-bit volume pointer %p is not 16-byte aligned", p);
    return FZ_OK;
}

}  // namespace

bool pairs_supported(const DevGeom& G, const fz_solver& s, int relu) {
    if (G.S < 2 || G.S % 2 || G.n[2] % 2) return false;
    int base[FZ_MAX_SHIFTS][3];
    if (!find_pairs(G, base)) return false;
    for (int q = 0; q < G.S / 2; ++q)
        if (base[q][2] % 2) return false;          // the roll kernels move voxel pairs
    return phase_supported(pair_geom(G), s, relu);
}

size_t pairs_saved_bytes(const DevGeom& G, const fz_solver& s) {
    return (size_t)G.S * G.mats_per_shift * (rec_head_for(s.num_iters) + 72) * sizeof(float);
}

size_t pairs_workspace_bytes(const DevGeom& G, const fz_solver& s) {
    const size_t f32_vols = G.dtype != FZ_DTYPE_F32 ? 2 : 1;
    return align_up(phase_workspace_bytes(pair_geom(G), s), 256) + 2 * vol_bytes(G, elem_bytes(G)) + f32_vols * vol_bytes(G, sizeof(float));
}

// Every pair's octant kernels write an fp32 partial sum (the unshifted pair's straight into the sum); a 16-bit volume's y is
// written once, by the last combine, so the partial sums are never rounded to 16 bits.
int pairs_forward(const float* x, const float* v0, float* y, void* saved, void* workspace, const DevGeom& G,
                  const fz_solver& s, cudaStream_t st) {
    if (!workspace) return fail(FZ_ERR_INVALID, "fz_swnmf_forward: workspace of %zu bytes required", pairs_workspace_bytes(G, s));
    const bool h16 = G.dtype != FZ_DTYPE_F32;
    if (h16) if (int e = check_16bit_pointers({x, y})) return e;
    const DevGeom Gp = pair_geom(G);
    int base[FZ_MAX_SHIFTS][3];
    find_pairs(G, base);
    const int np = G.S / 2;
    const PairBufs b = pair_bufs(workspace, G, s, y);
    const size_t saved_stride = (size_t)2 * Gp.mats_per_shift * (rec_head_for(s.num_iters) + 72) * sizeof(float);
    for (int k = 0; k < np; ++k) {
        const bool rolled = base[k][0] || base[k][1] || base[k][2];
        const float* xin = x;
        if (rolled) {
            if (int e = launch_roll(x, b.xr, G, base[k], st)) return e;
            xin = b.xr;
        }
        void* sv = saved ? static_cast<char*>(saved) + k * saved_stride : nullptr;
        if (!rolled && np == 1) return phase_forward(xin, v0, y, sv, workspace, Gp, s, st);
        const bool direct = !rolled && k == 0;       // the unshifted pair writes (the start of) the sum in place
        if (int e = phase_forward(xin, v0, direct ? b.acc : b.part, sv, workspace, Gp, s, st, true)) return e;
        const bool last = k == np - 1;
        if (!direct)
            if (int e = launch_combine(b.acc, b.part, G, base[k], k == 0, last ? 1.f / (float)np : 1.f, h16 && last ? y : nullptr, st))
                return e;
    }
    return FZ_OK;
}

int pairs_backward(const float* x, const float* gy, const float* v0, const void* saved, float* gx, void* workspace,
                   const DevGeom& G, const fz_solver& s, int K, cudaStream_t st) {
    if (!workspace) return fail(FZ_ERR_INVALID, "fz_swnmf_backward: workspace of %zu bytes required", pairs_workspace_bytes(G, s));
    if (!saved) return fail(FZ_ERR_INVALID, "fz_swnmf_backward: the `saved` buffer written by fz_swnmf_forward is required");
    const bool h16 = G.dtype != FZ_DTYPE_F32;
    if (h16) if (int e = check_16bit_pointers({x, gy, gx})) return e;
    const DevGeom Gp = pair_geom(G);
    int base[FZ_MAX_SHIFTS][3];
    find_pairs(G, base);
    const int np = G.S / 2;
    const PairBufs b = pair_bufs(workspace, G, s, gx);
    const size_t saved_stride = (size_t)2 * Gp.mats_per_shift * (rec_head_for(s.num_iters) + 72) * sizeof(float);
    for (int k = 0; k < np; ++k) {
        const bool rolled = base[k][0] || base[k][1] || base[k][2];
        const float *xin = x, *gin = gy;
        if (rolled) {
            if (int e = launch_roll(x, b.xr, G, base[k], st)) return e;
            if (int e = launch_roll(gy, b.gr, G, base[k], st)) return e;
            xin = b.xr; gin = b.gr;
        }
        const void* sv = static_cast<const char*>(saved) + k * saved_stride;
        if (!rolled && np == 1) return phase_backward(xin, gin, v0, sv, gx, workspace, Gp, s, K, st);
        const bool direct = !rolled && k == 0;
        if (int e = phase_backward(xin, gin, v0, sv, direct ? b.acc : b.part, workspace, Gp, s, K, st, true)) return e;
        const bool last = k == np - 1;
        if (!direct)
            if (int e = launch_combine(b.acc, b.part, G, base[k], k == 0, last ? 1.f / (float)np : 1.f, h16 && last ? gx : nullptr, st))
                return e;
    }
    return FZ_OK;
}

}  // namespace fz
