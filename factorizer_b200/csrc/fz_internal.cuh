// Cross-translation-unit declarations (not part of the C ABI).
#pragma once
#include "fz_common.cuh"

namespace fz {

struct NmfArgs {
    // forward
    const float* x;   // direct: (n,M,N); window: volume (B,C,D,H,W)
    const float* u0;  // (M,R)
    const float* v0;  // (N,R)
    float* u;         // (n,M,R) or null
    float* v;         // (n,N,R) or null
    float* y;         // direct: (n,M,N) or null; window: volume
    // backward
    const float* gy;  // direct (n,M,N) / window: volume
    const float* gu;  // (n,M,R) or null
    const float* gv;  // (n,N,R) or null
    float* gx;        // direct (n,M,N) / window: volume
    long long n;      // matrices handled by this launch
    int M, N, T, K, kind;
    float eps;
    // window mode
    DevGeom G;
    int shift;  // which window set this launch handles
    int relu;
    // direct mode only: X (and the gradient accumulator) stay in global memory -- matrices whose working set exceeds one CTA's
    // shared memory (set by the launcher)
    int spill;
};

// fz_nmf_generic.cu
int check_solver(const fz_solver* s, int M, int N, int* K);
int generic_direct(const NmfArgs& a, int R, bool bwd, cudaStream_t st);
int generic_window(NmfArgs a, int R, bool bwd, cudaStream_t st);

// fz_swnmf_fast.cu
bool fast_supported(const DevGeom& G, const fz_solver& s);
size_t fast_saved_bytes(const DevGeom& G, const fz_solver& s);
size_t fast_workspace_bytes(const DevGeom& G, const fz_solver& s);
int fast_forward(const float* x, const float* u0, const float* v0, float* y, void* saved,
                 void* workspace, const DevGeom& G, const fz_solver& s, int relu, cudaStream_t st);
int fast_backward(const float* x, const float* gy, const float* u0, const float* v0,
                  const void* saved, float* gx, void* workspace, const DevGeom& G,
                  const fz_solver& s, int K, int relu, cudaStream_t st);

// fz_swnmf_small.cu: rank-1 HALS / MU on small matrices (N = 64 with M = 4, 8, 16, 32; 8x16, 8x128, 8x256), a sub-warp each.
// Window mode takes fp32 or bf16 volumes; a bf16 volume at S >= 2 sums the window sets in an fp32 volume in the workspace
bool small_supported(int M, int N, const fz_solver& s);
bool small_window_supported(const DevGeom& G, const fz_solver& s);
size_t small_workspace_bytes(const DevGeom& G);
int small_direct(const float* x, const float* u0, const float* v0, const float* gy, float* out, long long n, int M, int N,
                 const fz_solver& s, int K, bool bwd, cudaStream_t st);
int small_window(const float* x, const float* u0, const float* v0, const float* gy, float* out, void* workspace,
                 const DevGeom& G, const fz_solver& s, int K, int relu, bool bwd, cudaStream_t st);

// fz_swnmf_phase.cu: three-pass "octant" formulation for [unshifted, shifted by patch/2], act = ReLU.  y / gx have the
// volume's element type, or fp32 with f32_out (the partial sums of the paired variant below)
bool phase_supported(const DevGeom& G, const fz_solver& s, int relu);
size_t phase_workspace_bytes(const DevGeom& G, const fz_solver& s);
int phase_forward(const float* x, const float* v0, float* y, void* saved, void* workspace,
                  const DevGeom& G, const fz_solver& s, cudaStream_t st, bool f32_out = false);
int phase_backward(const float* x, const float* gy, const float* v0, const void* saved, float* gx,
                   void* workspace, const DevGeom& G, const fz_solver& s, int K, cudaStream_t st, bool f32_out = false);

// fz_swnmf_pipe.cu: the same formulation as ONE persistent, software-pipelined launch per direction (large volumes)
bool pipe_supported(const DevGeom& G, const fz_solver& s, int relu, int force);
size_t pipe_workspace_bytes(const DevGeom& G, const fz_solver& s);
int pipe_forward(const float* x, const float* v0, float* y, void* saved, void* workspace,
                 const DevGeom& G, const fz_solver& s, cudaStream_t st);
int pipe_backward(const float* x, const float* gy, const float* v0, const void* saved, float* gx,
                  void* workspace, const DevGeom& G, const fz_solver& s, int K, cudaStream_t st);

// fz_block_glue_fwd_tc.cu: tcgen05 / TMEM versions of the two forward glue kernels (A operands in tensor memory, 3xTF32)
bool mixer_mlp_tc_supported(int hidden);
int mixer_mlp_tc_launch(const float* x, const float* m, const float* Wout, const float* bout, const float* gamma, const float* beta,
                        const float* W1, const float* b1, const float* W2, const float* b2, float* x1, float* out, long long batch,
                        int hidden, long long voxels, float eps, cudaStream_t st);
int ln_linear_tc_launch(const float* x, const float* gamma, const float* beta, const float* W, float* y, long long batch,
                        long long voxels, float eps, cudaStream_t st);

// fz_block_glue_lin_tc.cu: tcgen05 / TMEM version of linear_bwd (dgrad with A in tensor memory, weight gradient as a contraction
// over voxel rows); the caller zeroes the gradients
int linear_bwd_tc2_launch(const float* dy, const float* a, const float* gamma, const float* beta, const float* W, const float* resid,
                          float* da, float* dW, float* db, float* dgamma, float* dbeta, long long batch, long long voxels, float eps,
                          int layernorm, cudaStream_t st);

// fz_linear_tc.cu: weight gradient of a pointwise channel map on tcgen05 (any channel counts); the caller zeroes dW / db
bool linear_wgrad_tc_supported(const float* dy, const float* x, long long batch, int cout, int cin, long long voxels);
int linear_wgrad_tc_launch(const float* dy, const float* x, float* dW, float* db, long long batch, int cout, int cin, long long voxels,
                           cudaStream_t st);

bool linear_fwd_tc_supported(const float* x, const float* W, long long batch, int cout, int cin, long long voxels);
int linear_fwd_tc_launch(const float* x, const float* W, const float* bias, float* y, const float* aux, float* y2, int epi,
                         int wt, long long batch, int cout, int cin, long long voxels, cudaStream_t st);

// fz_block_glue_bwd_tc.cu: tcgen05 / TMEM version of the MLP + norm2 backward kernel (hidden width a multiple of 64, 3xTF32); the caller
// zeroes the gradients
bool mlp_bwd_tc_supported(int hidden);
int mlp_bwd_tc_launch(const float* x1, const float* dout, const float* gamma, const float* beta, const float* W1, const float* b1,
                      const float* W2, float* dx1, float* dgamma, float* dbeta, float* dW1, float* db1, float* dW2, float* db2,
                      long long batch, int hidden, long long voxels, float eps, cudaStream_t st);

// fz_nmf_big.cu: rank-1 MU / HALS on matrices too large for one CTA (global Matricize: M channels x all voxels), one
// grid-wide pass per sweep
bool big_supported(int M, long long N, const fz_solver& s);
size_t big_saved_bytes(long long n, int M, long long N, const fz_solver& s);
size_t big_workspace_bytes(long long n, int M, long long N, const fz_solver& s);
int big_forward(const float* x, const float* u0, const float* v0, float* y, void* saved, void* workspace, long long n, int M,
                long long N, const fz_solver& s, int relu, cudaStream_t st);
int big_backward(const float* x, const float* gy, const float* u0, const float* v0, const void* saved, float* gx,
                 void* workspace, long long n, int M, long long N, const fz_solver& s, int K, int relu, cudaStream_t st);

// ... and window sets that pair up as (a, a + patch/2): one octant problem per pair on the volume rolled by a
bool pairs_supported(const DevGeom& G, const fz_solver& s, int relu);
size_t pairs_saved_bytes(const DevGeom& G, const fz_solver& s);
size_t pairs_workspace_bytes(const DevGeom& G, const fz_solver& s);
int pairs_forward(const float* x, const float* v0, float* y, void* saved, void* workspace, const DevGeom& G,
                  const fz_solver& s, cudaStream_t st);
int pairs_backward(const float* x, const float* gy, const float* v0, const void* saved, float* gx, void* workspace,
                   const DevGeom& G, const fz_solver& s, int K, cudaStream_t st);

}  // namespace fz
