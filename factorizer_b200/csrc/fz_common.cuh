// Shared host/device helpers for the factorizer_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/factorizer_b200.h"

namespace fz {

// ---- error reporting ---------------------------------------------------------------------------
struct TlsState {
    char msg[512];
    int path;
    int launches;
    int glue_mode;   // fz_set_glue_mode() of the calling thread (all tensor-core paths on by default)
};
TlsState& tls();
int fail(int code, const char* fmt, ...);

// cuTensorMapEncodeTiled (driver entry point, looked up once) with element strides of 1, no interleave, L2 promotion in
// 128-byte lines and out-of-bounds elements read as zeros; every tensor map of the library is encoded here.  On failure:
// fail(FZ_ERR_CUDA, ...) naming the map (`what`).
int encode_tiled_map(CUtensorMap* m, const char* what, CUtensorMapDataType type, cuuint32_t rank, const void* ptr,
                     const cuuint64_t* dims, const cuuint64_t* strides, const cuuint32_t* box, CUtensorMapSwizzle swizzle);

#define FZ_CUDA_CHECK(expr)                                                                     \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess)                                                                  \
            return ::fz::fail(FZ_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                              __FILE__, __LINE__);                                              \
    } while (0)

#define FZ_LAUNCH_CHECK()                                                                       \
    do {                                                                                        \
        ::fz::tls().launches++;                                                                 \
        FZ_CUDA_CHECK(cudaGetLastError());                                                      \
    } while (0)

// Per-device high-water mark of the dynamic shared memory a kernel has been configured for
// (cudaFuncSetAttribute applies to the current device only).  Not synchronised: the worst case is a repeated,
// idempotent attribute call.
struct SmemConfig {
    size_t bytes[64] = {0};
    template <typename K>
    cudaError_t ensure(K kernel, size_t need) {
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        size_t& have = bytes[dev & 63];
        if (need <= have) return cudaSuccess;
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need);
        if (e == cudaSuccess) have = need;
        return e;
    }
};

// Number of SMs of the CURRENT device (cached per device; a process may drive several GPUs).
inline int num_sms() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    int& v = cached[dev & 63];
    if (v <= 0) {
        int sms = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        v = sms > 0 ? sms : 148;
    }
    return v;
}

// ---- device-side geometry ----------------------------------------------------------------------
// Derived from fz_geom once on the host; passed to kernels by value.
struct DevGeom {
    int B, C, heads, d;      // batch, channels, C/d, head_dim (= M)
    int n[3];                // D, H, W
    int p[3];                // patch
    int g[3];                // grid = n / p
    int S;                   // number of window sets
    int sh[FZ_MAX_SHIFTS][3];
    int G;                   // windows per (batch, head): g0*g1*g2
    int P;                   // columns per matrix: p0*p1*p2 (= N)
    long long vox;           // D*H*W
    long long mats_per_shift;  // B*heads*G
    int path;                // fz_geom.path (FZ_PATH_*)
    int dtype;               // fz_geom.dtype (FZ_DTYPE_*): element type of the volumes
};

int make_dev_geom(const fz_geom* g, DevGeom* out);

// Offset (in elements, relative to channel 0 of batch 0) of column j of window w under shift set s:
// x[(g_k*p_k + q_k - sh_k) mod n_k]  (torch.roll: rolled[i] = x[(i - shift) mod n],
// factorizer/factorization/operations.py:268-269).
__device__ __forceinline__ long long window_col_offset(const DevGeom& G, int s, int w, int j) {
    int g2 = w % G.g[2];
    int t = w / G.g[2];
    int g1 = t % G.g[1];
    int g0 = t / G.g[1];
    int q2 = j % G.p[2];
    t = j / G.p[2];
    int q1 = t % G.p[1];
    int q0 = t / G.p[1];
    int i0 = g0 * G.p[0] + q0 - G.sh[s][0];
    int i1 = g1 * G.p[1] + q1 - G.sh[s][1];
    int i2 = g2 * G.p[2] + q2 - G.sh[s][2];
    i0 %= G.n[0]; if (i0 < 0) i0 += G.n[0];
    i1 %= G.n[1]; if (i1 < 0) i1 += G.n[1];
    i2 %= G.n[2]; if (i2 < 0) i2 += G.n[2];
    return ((long long)i0 * G.n[1] + i1) * G.n[2] + i2;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace fz
