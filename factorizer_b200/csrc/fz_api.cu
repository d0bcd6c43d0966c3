// extern "C" entry points: argument validation, error strings, kernel selection.
#include <string.h>

#include "fz_common.cuh"
#include "fz_internal.cuh"

namespace fz {

TlsState& tls() {
    static thread_local TlsState s = {{0}, 0, 0, 7};
    return s;
}

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(tls().msg, sizeof(tls().msg), fmt, ap);
    va_end(ap);
    return code;
}

int encode_tiled_map(CUtensorMap* m, const char* what, CUtensorMapDataType type, cuuint32_t rank, const void* ptr,
                     const cuuint64_t* dims, const cuuint64_t* strides, const cuuint32_t* box, CUtensorMapSwizzle swizzle) {
    typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                      const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeTiledFn enc = nullptr;
    if (!enc) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            enc = reinterpret_cast<EncodeTiledFn>(p);
    }
    if (!enc) return fail(FZ_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
    // the driver call needs the device's context current on the calling thread; a thread that has made no runtime call yet
    // (autograd's backward thread, when a tensor map is its first CUDA work) has none
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaSetDevice(dev) != cudaSuccess) return fail(FZ_ERR_CUDA, "no usable CUDA device");
    const cuuint32_t es[5] = {1, 1, 1, 1, 1};
    const CUresult r = enc(m, type, rank, const_cast<void*>(ptr), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(FZ_ERR_CUDA, "cuTensorMapEncodeTiled (%s) failed with CUresult %d", what, (int)r);
    return FZ_OK;
}

// One window per (sample, head), no roll, and more elements than a CTA can hold: Matricize(grid_size=1), the
// reference's default FactMixer reshape (factorizer/factorizer.py:17).  The matrix is the contiguous block
// x[b, h*d:(h+1)*d, :].
static bool big_window(const DevGeom& G, const fz_solver& s) {
    if (G.G != 1 || G.S != 1) return false;
    for (int k = 0; k < 3; ++k)
        if (G.sh[0][k] % G.n[k]) return false;
    return (long long)G.d * G.P >= 16384 && big_supported(G.d, G.P, s);
}

int make_dev_geom(const fz_geom* g, DevGeom* o) {
    if (!g) return fail(FZ_ERR_INVALID, "null geometry");
    if (g->batch < 0 || g->channels < 1 || g->head_dim < 1)
        return fail(FZ_ERR_INVALID, "bad geometry: batch=%d channels=%d head_dim=%d", g->batch,
                    g->channels, g->head_dim);
    if (g->channels % g->head_dim)
        return fail(FZ_ERR_INVALID, "channels=%d not divisible by head_dim=%d", g->channels, g->head_dim);
    if (g->num_shifts < 1 || g->num_shifts > FZ_MAX_SHIFTS)
        return fail(FZ_ERR_UNSUPPORTED, "num_shifts=%d outside 1..%d", g->num_shifts, FZ_MAX_SHIFTS);
    o->B = g->batch;
    o->C = g->channels;
    o->d = g->head_dim;
    o->heads = g->channels / g->head_dim;
    o->S = g->num_shifts;
    o->vox = 1;
    o->G = 1;
    o->P = 1;
    for (int k = 0; k < 3; ++k) {
        if (g->size[k] < 1 || g->patch[k] < 1 || g->size[k] % g->patch[k])
            return fail(FZ_ERR_INVALID, "size[%d]=%d not divisible by patch[%d]=%d", k, g->size[k], k,
                        g->patch[k]);
        o->n[k] = g->size[k];
        o->p[k] = g->patch[k];
        o->g[k] = g->size[k] / g->patch[k];
        o->vox *= g->size[k];
        o->G *= o->g[k];
        o->P *= o->p[k];
    }
    if (o->vox >= (1LL << 31)) return fail(FZ_ERR_UNSUPPORTED, "volume of %lld voxels too large", o->vox);
    for (int s = 0; s < FZ_MAX_SHIFTS; ++s)
        for (int k = 0; k < 3; ++k) o->sh[s][k] = s < g->num_shifts ? g->shifts[s][k] : 0;
    o->mats_per_shift = (long long)o->B * o->heads * o->G;
    if (g->path < FZ_PATH_AUTO || g->path > FZ_PATH_OCTANT_PIPELINE)
        return fail(FZ_ERR_INVALID, "fz_geom.path=%d is not one of FZ_PATH_*", g->path);
    o->path = g->path;
    if (g->dtype != FZ_DTYPE_F32 && g->dtype != FZ_DTYPE_BF16 && g->dtype != FZ_DTYPE_F16)
        return fail(FZ_ERR_INVALID, "fz_geom.dtype=%d is not one of FZ_DTYPE_*", g->dtype);
    o->dtype = g->dtype;
    return FZ_OK;
}

}  // namespace fz

using namespace fz;

extern "C" {

int fz_version(void) { return FZ_VERSION; }
const char* fz_last_error(void) { return tls().msg; }
int fz_last_path(void) { return tls().path; }
int fz_last_launches(void) { return tls().launches; }

int fz_nmf_forward(const float* x, const float* u0, const float* v0, float* u, float* v, float* y,
                   int64_t n, int32_t M, int32_t N, const fz_solver* s, void* stream) {
    tls().launches = 0;
    tls().path = 0;
    int K;
    if (int e = check_solver(s, M, N, &K)) return e;
    if (n < 0) return fail(FZ_ERR_INVALID, "n=%lld < 0", (long long)n);
    if (!x || !u0 || !v0) return fail(FZ_ERR_INVALID, "null input buffer");
    if (y && !u && !v && small_supported(M, N, *s)) {
        tls().path = 3;
        return small_direct(x, u0, v0, nullptr, y, n, M, N, *s, K, false, (cudaStream_t)stream);
    }
    NmfArgs a;
    memset(&a, 0, sizeof(a));
    a.x = x; a.u0 = u0; a.v0 = v0; a.u = u; a.v = v; a.y = y;
    a.n = n; a.M = M; a.N = N; a.T = s->num_iters; a.K = K; a.kind = s->kind; a.eps = s->eps;
    return generic_direct(a, s->rank, false, (cudaStream_t)stream);
}

int fz_nmf_backward(const float* x, const float* u0, const float* v0, const float* gy,
                    const float* gu, const float* gv, float* gx, int64_t n, int32_t M, int32_t N,
                    const fz_solver* s, void* stream) {
    tls().launches = 0;
    tls().path = 0;
    int K;
    if (int e = check_solver(s, M, N, &K)) return e;
    if (n < 0) return fail(FZ_ERR_INVALID, "n=%lld < 0", (long long)n);
    if (!x || !u0 || !v0 || !gx) return fail(FZ_ERR_INVALID, "null buffer");
    if (gy && !gu && !gv && small_supported(M, N, *s)) {
        tls().path = 3;
        return small_direct(x, u0, v0, gy, gx, n, M, N, *s, K, true, (cudaStream_t)stream);
    }
    NmfArgs a;
    memset(&a, 0, sizeof(a));
    a.x = x; a.u0 = u0; a.v0 = v0; a.gy = gy; a.gu = gu; a.gv = gv; a.gx = gx;
    a.n = n; a.M = M; a.N = N; a.T = s->num_iters; a.K = K; a.kind = s->kind; a.eps = s->eps;
    return generic_direct(a, s->rank, true, (cudaStream_t)stream);
}

size_t fz_swnmf_saved_bytes(const fz_geom* g, const fz_solver* s) {
    DevGeom G;
    if (make_dev_geom(g, &G) || !s) return 0;
    // The caller does not say here whether the input passes through a ReLU, so size the buffer for whichever
    // kernel family fz_swnmf_forward may pick for this geometry (the octant kernels and their paired variant have
    // no limit on the number of windows, the window-at-a-time kernels do).
    size_t need = fast_saved_bytes(G, *s);
    if (phase_supported(G, *s, 1) || pairs_supported(G, *s, 1)) {
        const size_t b = pairs_saved_bytes(G, *s);      // S * windows * record, the same record for both
        if (b > need) need = b;
    }
    if (big_window(G, *s)) {
        const size_t b = big_saved_bytes(G.mats_per_shift, G.d, G.P, *s);
        if (b > need) need = b;
    }
    return need;
}

size_t fz_swnmf_workspace_bytes(const fz_geom* g, const fz_solver* s) {
    DevGeom G;
    if (make_dev_geom(g, &G) || !s) return 0;
    size_t a = fast_workspace_bytes(G, *s);
    if (phase_supported(G, *s, 1)) {
        size_t b = phase_workspace_bytes(G, *s);
        if (b > a) a = b;
        if (pipe_supported(G, *s, 1, 1)) {
            b = pipe_workspace_bytes(G, *s);
            if (b > a) a = b;
        }
    } else if (pairs_supported(G, *s, 1)) {
        const size_t b = pairs_workspace_bytes(G, *s);
        if (b > a) a = b;
    }
    if (small_window_supported(G, *s)) {
        const size_t b = small_workspace_bytes(G);
        if (b > a) a = b;
    }
    if (big_window(G, *s)) {
        const size_t b = big_workspace_bytes(G.mats_per_shift, G.d, G.P, *s);
        if (b > a) a = b;
    }
    return a;
}

static const char* const k16BitCoverage =
    "bf16 and fp16 volumes are served by the octant kernels (head_dim 8, patch 8x8x8, ReLU, rank-1 HALS, an even number of "
    "patches along W, and window sets that pair up as (a, a + 4) with every base shift a even along W, e.g. shifts "
    "[0, 4] or [0, 2, 4, 6]) and by the sub-warp kernels (64-column windows with head_dim 4, 8, 16 or 32, or 8 x 16, "
    "8 x 128 or 8 x 256 windows, at any shifts, rank-1 HALS or MU with up to 5 iterations, ReLU or not)";

// The window-at-a-time 8x512 kernels (path 1), the grid-wide (5) and the generic (0) kernels take fp32 volumes only.
static bool half_small_ok(const DevGeom& G, const fz_solver& s) {
    return G.path != FZ_PATH_GENERIC && small_window_supported(G, s);
}

// bf16 and fp16 volumes take the same kernels at the same geometries
static int half_supported(const fz_geom* g, const fz_solver* s, int32_t relu_input, int dtype) {
    if (!g || !s) return 0;
    fz_geom gb = *g;
    gb.dtype = dtype;
    DevGeom G;
    int K;
    if (make_dev_geom(&gb, &G) || check_solver(s, G.d, G.P, &K)) return 0;
    return phase_supported(G, *s, relu_input) || pairs_supported(G, *s, relu_input) || half_small_ok(G, *s) ? 1 : 0;
}

int fz_swnmf_bf16_supported(const fz_geom* g, const fz_solver* s, int32_t relu_input) {
    return half_supported(g, s, relu_input, FZ_DTYPE_BF16);
}

int fz_swnmf_f16_supported(const fz_geom* g, const fz_solver* s, int32_t relu_input) {
    return half_supported(g, s, relu_input, FZ_DTYPE_F16);
}

int fz_swnmf_forward(const float* x, const float* u0, const float* v0, float* y, void* saved,
                     void* workspace, const fz_geom* g, const fz_solver* s, int32_t relu_input,
                     void* stream) {
    tls().launches = 0;
    DevGeom G;
    if (int e = make_dev_geom(g, &G)) return e;
    int K;
    if (int e = check_solver(s, G.d, G.P, &K)) return e;
    if (G.B == 0) return FZ_OK;                       // empty batch: tensors carry null data pointers
    if (!x || !u0 || !v0 || !y) return fail(FZ_ERR_INVALID, "null buffer");
    const bool octant_ok = G.path == FZ_PATH_AUTO || G.path == FZ_PATH_OCTANT_3LAUNCH || G.path == FZ_PATH_OCTANT_PIPELINE;
    const bool fast_ok = G.path != FZ_PATH_GENERIC;
    if (octant_ok && G.path != FZ_PATH_OCTANT_3LAUNCH && pipe_supported(G, *s, relu_input, G.path == FZ_PATH_OCTANT_PIPELINE)) {
        tls().path = 6;
        return pipe_forward(x, v0, y, saved, workspace, G, *s, (cudaStream_t)stream);
    }
    if (octant_ok && phase_supported(G, *s, relu_input)) {
        tls().path = 2;
        return phase_forward(x, v0, y, saved, workspace, G, *s, (cudaStream_t)stream);
    }
    if (octant_ok && pairs_supported(G, *s, relu_input)) {
        tls().path = 4;
        const int e = pairs_forward(x, v0, y, saved, workspace, G, *s, (cudaStream_t)stream);
        tls().path = 4;
        return e;
    }
    if (G.dtype != FZ_DTYPE_F32) {
        if (!half_small_ok(G, *s)) return fail(FZ_ERR_UNSUPPORTED, "%s", k16BitCoverage);
        tls().path = 3;
        return small_window(x, u0, v0, nullptr, y, workspace, G, *s, K, relu_input, false, (cudaStream_t)stream);
    }
    if (fast_ok && fast_supported(G, *s)) {
        tls().path = 1;
        return fast_forward(x, u0, v0, y, saved, workspace, G, *s, relu_input, (cudaStream_t)stream);
    }
    if (fast_ok && small_window_supported(G, *s)) {
        tls().path = 3;
        return small_window(x, u0, v0, nullptr, y, workspace, G, *s, K, relu_input, false, (cudaStream_t)stream);
    }
    if (big_window(G, *s)) {
        tls().path = 5;
        return big_forward(x, u0, v0, y, saved, workspace, G.mats_per_shift, G.d, G.P, *s, relu_input, (cudaStream_t)stream);
    }
    tls().path = 0;
    NmfArgs a;
    memset(&a, 0, sizeof(a));
    a.x = x; a.u0 = u0; a.v0 = v0; a.y = y;
    a.n = G.mats_per_shift; a.M = G.d; a.N = G.P; a.T = s->num_iters; a.K = K; a.kind = s->kind;
    a.eps = s->eps; a.G = G; a.relu = relu_input;
    return generic_window(a, s->rank, false, (cudaStream_t)stream);
}

int fz_swnmf_backward(const float* x, const float* gy, const float* u0, const float* v0,
                      const void* saved, float* gx, void* workspace, const fz_geom* g,
                      const fz_solver* s, int32_t relu_input, void* stream) {
    tls().launches = 0;
    DevGeom G;
    if (int e = make_dev_geom(g, &G)) return e;
    int K;
    if (int e = check_solver(s, G.d, G.P, &K)) return e;
    if (G.B == 0) return FZ_OK;
    if (!x || !gy || !u0 || !v0 || !gx) return fail(FZ_ERR_INVALID, "null buffer");
    const bool octant_ok = G.path == FZ_PATH_AUTO || G.path == FZ_PATH_OCTANT_3LAUNCH || G.path == FZ_PATH_OCTANT_PIPELINE;
    const bool fast_ok = G.path != FZ_PATH_GENERIC;
    if (octant_ok && G.path != FZ_PATH_OCTANT_3LAUNCH && pipe_supported(G, *s, relu_input, G.path == FZ_PATH_OCTANT_PIPELINE)) {
        tls().path = 6;
        return pipe_backward(x, gy, v0, saved, gx, workspace, G, *s, K, (cudaStream_t)stream);
    }
    if (octant_ok && phase_supported(G, *s, relu_input)) {
        tls().path = 2;
        return phase_backward(x, gy, v0, saved, gx, workspace, G, *s, K, (cudaStream_t)stream);
    }
    if (octant_ok && pairs_supported(G, *s, relu_input)) {
        tls().path = 4;
        return pairs_backward(x, gy, v0, saved, gx, workspace, G, *s, K, (cudaStream_t)stream);
    }
    if (G.dtype != FZ_DTYPE_F32) {
        if (!half_small_ok(G, *s)) return fail(FZ_ERR_UNSUPPORTED, "%s", k16BitCoverage);
        tls().path = 3;
        return small_window(x, u0, v0, gy, gx, workspace, G, *s, K, relu_input, true, (cudaStream_t)stream);
    }
    if (fast_ok && fast_supported(G, *s)) {
        tls().path = 1;
        return fast_backward(x, gy, u0, v0, saved, gx, workspace, G, *s, K, relu_input,
                             (cudaStream_t)stream);
    }
    if (fast_ok && small_window_supported(G, *s)) {
        tls().path = 3;
        return small_window(x, u0, v0, gy, gx, workspace, G, *s, K, relu_input, true, (cudaStream_t)stream);
    }
    if (big_window(G, *s)) {
        tls().path = 5;
        return big_backward(x, gy, u0, v0, saved, gx, workspace, G.mats_per_shift, G.d, G.P, *s, K, relu_input,
                            (cudaStream_t)stream);
    }
    tls().path = 0;
    NmfArgs a;
    memset(&a, 0, sizeof(a));
    a.x = x; a.gy = gy; a.u0 = u0; a.v0 = v0; a.gx = gx;
    a.n = G.mats_per_shift; a.M = G.d; a.N = G.P; a.T = s->num_iters; a.K = K; a.kind = s->kind;
    a.eps = s->eps; a.G = G; a.relu = relu_input;
    return generic_window(a, s->rank, true, (cudaStream_t)stream);
}

}  // extern "C"
