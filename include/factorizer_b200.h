/*
 * factorizer_b200 -- C ABI of the B200-native (sm_100a) Factorizer hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  Every entry point
 * replaces a piece of the reference's (pashtari/factorizer) PyTorch eager path; the reference
 * interface it stands in for is cited as file:line relative to the reference checkout.
 *
 * Conventions
 *   - all data pointers are DEVICE pointers to C-contiguous float32 buffers on the current device;
 *     the caller owns every buffer, the library never allocates user-visible memory;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); every call is
 *     asynchronous on that stream, performs no host synchronisation and is CUDA-graph capturable;
 *   - return value 0 = success, otherwise one of FZ_ERR_*; a thread-local message is available from
 *     fz_last_error().  No C++ exception crosses this boundary;
 *   - volumes are (B, C, D, H, W) = NCDHW; inputs with fewer than three spatial dims pad
 *     size/patch/shifts on the LEFT with 1/1/0;
 *   - matricised tensors are (S*B*heads, G, d, P) with row index s*(B*heads) + b*heads + h,
 *     window index (g0*G1+g1)*G2+g2, row dd (channel h*d+dd), column (q0*P1+q1)*P2+q2
 *     (factorizer/factorization/operations.py:321-325, 417-421).
 */
#ifndef FACTORIZER_B200_H_
#define FACTORIZER_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FZ_VERSION 100          /* 0.1.0 */
#define FZ_MAX_SHIFTS 8
#define FZ_MAX_RANK 8

enum {
    FZ_OK = 0,
    FZ_ERR_INVALID = 1,         /* malformed argument (null pointer, non-divisible geometry, ...) */
    FZ_ERR_UNSUPPORTED = 2,     /* valid but outside what the kernels implement                    */
    FZ_ERR_CUDA = 3             /* CUDA runtime / driver error (message carries cudaGetErrorString) */
};

enum { FZ_SOLVER_MU = 0, FZ_SOLVER_HALS = 1 };
enum { FZ_DTYPE_F32 = 0, FZ_DTYPE_BF16 = 1, FZ_DTYPE_F16 = 2 };

/* Window geometry of Matricize / SWMatricize
 * (factorizer/factorization/operations.py:299-355 and :381-415). */
typedef struct fz_geom {
    int32_t batch;                      /* B                                                   */
    int32_t channels;                   /* C = heads * head_dim                                */
    int32_t size[3];                    /* D, H, W                                             */
    int32_t patch[3];                   /* p0, p1, p2 (each must divide size)                  */
    int32_t head_dim;                   /* d = rows M of every matrix                          */
    int32_t num_shifts;                 /* S (1 for a plain Matricize)                         */
    int32_t shifts[FZ_MAX_SHIFTS][3];   /* torch.roll shifts per window set; 0 = unshifted     */
    int32_t dtype;                      /* FZ_DTYPE_F32 (0), FZ_DTYPE_BF16 or FZ_DTYPE_F16: element type of the VOLUMES
                                           handed to fz_swnmf_forward / _backward (x, y, dy, dx); u0, v0, the saved
                                           records and all arithmetic stay fp32, and a 16-bit y / dx is the fp32 result
                                           rounded once.  bf16 and fp16 are served by the octant kernels
                                           (head_dim 8, patch 8^3, ReLU, rank-1 HALS, an even number of patches along
                                           W) at shifts [0, 4] or at window sets that pair up as (a, a + 4) with even
                                           base shifts along W, e.g. [0, 2, 4, 6]; and by the sub-warp kernels at
                                           64-column windows with head_dim 4..32 (e.g. patch 4^3) and 8 x 16 / 128 /
                                           256 windows, at any shifts, rank-1 HALS or MU, up to 5 iterations, ReLU
                                           or not.  Anything else returns FZ_ERR_UNSUPPORTED                        */
    int32_t path;                       /* FZ_PATH_AUTO (0), or one of FZ_PATH_* to restrict the
                                           kernel family fz_swnmf_* may pick for this call (tests
                                           and measurements; a per-call argument, no global state) */
} fz_geom;

/* fz_geom.path: which kernel families fz_swnmf_forward / _backward may use.  The value is part of the call, so a
 * forward and its backward (which autograd may run on another thread) agree by construction. */
enum {
    FZ_PATH_AUTO = 0,            /* the fastest family that covers the geometry                               */
    FZ_PATH_GENERIC = 1,         /* one CTA per matrix out of shared memory only                              */
    FZ_PATH_NO_OCTANT = 2,       /* anything but the octant kernels (window-at-a-time / sub-warp / generic)   */
    FZ_PATH_OCTANT_3LAUNCH = 3,  /* octant kernels as three launches per direction, never the pipelined one   */
    FZ_PATH_OCTANT_PIPELINE = 4  /* octant kernels as one persistent launch per direction, whatever the size  */
};

/* The unrolled solver of MatrixFactorization.decompose
 * (factorizer/factorization/matrix_factorization.py:461-530). */
typedef struct fz_solver {
    int32_t kind;                       /* FZ_SOLVER_MU (:241-247) or FZ_SOLVER_HALS (:210-229) */
    int32_t rank;                       /* R, 1..FZ_MAX_RANK                                    */
    int32_t num_iters;                  /* T                                                    */
    int32_t num_grad_steps;             /* k: backward differentiates the last k iterations
                                           (context(), :506-512); <0 or >T means T             */
    float eps;                          /* 1e-16 (:200, :236)                                   */
} fz_solver;

int fz_version(void);
const char* fz_last_error(void);

/* ---- SWMatricize / Matricize, standalone and bit-exact ------------------------------------- */

/* SWMatricize.forward (operations.py:417-421; Reshape.forward :266-272):
 * x (B,C,D,H,W) -> y (S*B*heads, G, d, P).  Pure data movement. */
int fz_swmat_forward(const float* x, float* y, const fz_geom* g, void* stream);

/* SWMatricize.inverse_forward (operations.py:423-434; Reshape.inverse_forward :274-280):
 * out = ((0.0 + inv_0) + inv_1 + ...) / S, summed in shift order, then one true division. */
int fz_swmat_inverse(const float* y, float* x_out, const fz_geom* g, void* stream);

/* Adjoint of fz_swmat_forward: gx = sum_s unmatricize_s(gy_s) (what autograd's CatBackward /
 * RollBackward / permute chain computes for operations.py:417-421). */
int fz_swmat_forward_adjoint(const float* gy, float* gx, const fz_geom* g, void* stream);

/* Adjoint of fz_swmat_inverse: gy_s = matricize_s(g_out / S). */
int fz_swmat_inverse_adjoint(const float* g_out, float* gy, const fz_geom* g, void* stream);

/* ---- NMF on already-matricised tensors ------------------------------------------------------ */

/* MatrixFactorization.decompose + reconstruct (matrix_factorization.py:514-533, 544-546) with
 * RandomInit buffers (:28-58) broadcast to all `n` matrices.
 * x (n,M,N); u0 (M,R); v0 (N,R); outputs u (n,M,R), v (n,N,R), y (n,M,N) -- each may be NULL. */
int fz_nmf_forward(const float* x, const float* u0, const float* v0, float* u, float* v, float* y,
                   int64_t n, int32_t M, int32_t N, const fz_solver* s, void* stream);

/* dL/dx through the unrolled solver (replaces autograd's replay of the bmm/add/div/relu graph).
 * gy = dL/d(u v^T) (n,M,N), gu = dL/du (n,M,R), gv = dL/dv (n,N,R): any subset may be NULL. */
int fz_nmf_backward(const float* x, const float* u0, const float* v0, const float* gy,
                    const float* gu, const float* gv, float* gx, int64_t n, int32_t M, int32_t N,
                    const fz_solver* s, void* stream);

/* ---- fused FactMixer core: reshape -> act -> factorize -> inverse (factorizer.py:41-50) ----- */

/* Bytes of the `saved` buffer fz_swnmf_forward fills for fz_swnmf_backward (per-window iterate
 * summaries), and of the scratch `workspace` both directions need (tile-order counters; for bf16
 * and fp16 volumes on the sub-warp kernels with two or more window sets, an fp32 sum over the sets). */
size_t fz_swnmf_saved_bytes(const fz_geom* g, const fz_solver* s);
size_t fz_swnmf_workspace_bytes(const fz_geom* g, const fz_solver* s);

/* y_vol = SWMatricize.inverse_forward(NMF(act(SWMatricize(x_vol)))), act = ReLU if relu_input.
 * x, y: (B,C,D,H,W).  `saved` may be NULL when no backward will follow. */
int fz_swnmf_forward(const float* x, const float* u0, const float* v0, float* y, void* saved,
                     void* workspace, const fz_geom* g, const fz_solver* s, int32_t relu_input,
                     void* stream);

/* gx_vol = d<gy_vol, y_vol>/dx_vol.  `saved` is the buffer written by the matching forward (NULL
 * forces a full recompute of the iterates). */
int fz_swnmf_backward(const float* x, const float* gy, const float* u0, const float* v0,
                      const void* saved, float* gx, void* workspace, const fz_geom* g,
                      const fz_solver* s, int32_t relu_input, void* stream);

/* ---- channels-first LayerNorm: the glue on either side of the mixer (SURVEY section 8(f) row 1) ---- */

/* LayerNorm over the channel axis of a (batch, channels, voxels) tensor
 * (factorizer/layers/norm.py:25-34: movedim -> nn.LayerNorm(channels) -> movedim; biased variance, eps
 * inside the square root).  gamma / beta may be NULL (no affine).  Any channel count up to 512 (8, 16, 32 keep
 * all channels of a voxel in registers, the others loop) and an even number of voxels;
 * fz_layernorm_cf_supported() tells. */
int fz_layernorm_cf_supported(int32_t channels, int64_t voxels);
int fz_layernorm_cf_forward(const float* x, const float* gamma, const float* beta, float* y, int64_t batch,
                            int32_t channels, int64_t voxels, float eps, void* stream);
/* dx, and d(gamma), d(beta) (each `channels` floats, overwritten; either may be NULL) of <dy, y>. */
int fz_layernorm_cf_backward(const float* x, const float* gamma, const float* dy, float* dx, float* dgamma,
                             float* dbeta, int64_t batch, int32_t channels, int64_t voxels, float eps, void* stream);
/* the same with a residual gradient: dx = add + LN'(dy)  (the block's x + f(norm(x)) pattern, reference
 * factorizer/factorizer.py:74-77: one pass instead of LayerNorm backward + an elementwise sum); add may be NULL, must not
 * alias dx. */
int fz_layernorm_cf_backward_add(const float* x, const float* gamma, const float* dy, const float* add, float* dx,
                                 float* dgamma, float* dbeta, int64_t batch, int32_t channels, int64_t voxels, float eps,
                                 void* stream);

/* ---- weight gradient of the pointwise channel map (reference factorizer/layers/linear.py:53-58, a k=1 Conv1d) ----
 * dW[o][i] = sum over batch and voxels of dy[b][o][v] x[b][i][v]   (cout x cin floats, OVERWRITTEN)
 * db[o]    = sum over batch and voxels of dy[b][o][v]              (cout floats, OVERWRITTEN; may be NULL)
 * dy is (batch, cout, voxels), x is (batch, cin, voxels), fp32 contiguous.  voxels must be a multiple of 4 (channel
 * counts are free: blocks of 32 x 32 are zero-padded); fz_linear_wgrad_supported() tells.  dy and x must be 16-byte aligned
 * (FZ_ERR_UNSUPPORTED otherwise, before anything is written).  Replaces the large-K library SGEMM autograd picks for the
 * 64..512-channel stages of the Swin Factorizer. */
int fz_linear_wgrad_supported(int32_t cout, int32_t cin, int64_t voxels);
int fz_linear_wgrad(const float* dy, const float* x, float* dW, float* db, int64_t batch, int32_t cout, int32_t cin,
                    int64_t voxels, void* stream);

/* ---- the pointwise channel map itself (reference factorizer/layers/linear.py:53-58) on the tensor cores ----
 * y[b][o][v] = sum_i W[o][i] x[b][i][v] + bias[o]   (bias may be NULL); x is (batch, cin, voxels), y (batch, cout, voxels),
 * W (cout, cin) row-major, fp32 contiguous.  With W^T (cin, cout) and dy in place of x it is the input gradient.  3xTF32 on
 * tcgen05 (fp32 parity), for the wide stages whose library SGEMMs run on the FP32 pipe.  voxels and cin must be multiples of
 * 4, the pointers 16-byte aligned: fz_linear_forward_supported() tells. */
int fz_linear_forward_supported(int32_t cout, int32_t cin, int64_t voxels);
int fz_linear_forward(const float* x, const float* W, const float* bias, float* y, int64_t batch, int32_t cin, int32_t cout,
                      int64_t voxels, void* stream);
/* the same with a fused epilogue on r = W x + bias (same shapes as y for aux / y2):
 *   FZ_EPILOGUE_RESIDUAL   y = r + aux                      (x + out_proj(..), x1 + fc2(..): reference factorizer.py:74-77)
 *   FZ_EPILOGUE_GELU       y = r, y2 = gelu(r)  (exact erf)  (fc1 -> GELU, reference layers/mlp.py:54-60; r is kept for the backward)
 *   FZ_EPILOGUE_GELU_GRAD  y = r * gelu'(aux)               (the input gradient of fc2 through the GELU; aux = the saved r of fc1)
 *   FZ_EPILOGUE_GELU_ONLY  y = gelu(r)                      (inference: the pre-activation is not kept)
 * so that no elementwise pass is left between the channel maps of a block.  w_transposed != 0: W points to a (cin, cout)
 * row-major matrix and r = W^T x + bias -- the input gradient of a layer straight from its weight as stored (cout must be a
 * multiple of 4 then). */
enum { FZ_EPILOGUE_NONE = 0, FZ_EPILOGUE_RESIDUAL = 1, FZ_EPILOGUE_GELU = 2, FZ_EPILOGUE_GELU_GRAD = 3, FZ_EPILOGUE_GELU_ONLY = 4 };
int fz_linear_forward_ex(const float* x, const float* W, const float* bias, float* y, int64_t batch, int32_t cin, int32_t cout,
                         int64_t voxels, int32_t epilogue, int32_t w_transposed, const float* aux, float* y2, void* stream);

/* ---- bf16 activations (the FactorizerBlock under bf16 autocast, or fed bf16 tensors) -------------------------------------
 * Buffers typed `void*` below hold bf16 (torch.bfloat16) values; parameters, their gradients and the LayerNorm statistics
 * stay fp32, and every sum accumulates in fp32.  The bf16 TMA boxes need 16-byte row strides, so voxel counts must be
 * multiples of 8, and the buffers TMA reads (x, W, dy) 16-byte aligned: FZ_ERR_UNSUPPORTED otherwise, before anything
 * is written. */

/* fz_linear_forward_ex on bf16 activations: r = W x + bias with the same FZ_EPILOGUE_* (aux, y, y2 bf16; bias fp32, may be
 * NULL), applied to the fp32 sums before the one rounding to bf16.  W is a bf16 (cout, cin) matrix whose rows are ldw
 * elements apart (ldw >= cin, a multiple of 8), K-major; the input gradient passes the transposed copy written by
 * fz_bf16_stage_weights.  tcgen05 kind::f16, one MMA per 16 input channels. */
int fz_linear_forward_bf16_supported(int32_t cout, int32_t cin, int64_t voxels);
int fz_linear_forward_bf16(const void* x, const void* W, int32_t ldw, const float* bias, void* y, int64_t batch, int32_t cin,
                           int32_t cout, int64_t voxels, int32_t epilogue, const void* aux, void* y2, void* stream);
/* fz_linear_wgrad on bf16 dy (batch, cout, voxels) and x (batch, cin, voxels): dW (cout x cin) and db (cout, may be NULL)
 * fp32, OVERWRITTEN. */
int fz_linear_wgrad_bf16_supported(int32_t cout, int32_t cin, int64_t voxels);
int fz_linear_wgrad_bf16(const void* dy, const void* x, float* dW, float* db, int64_t batch, int32_t cout, int32_t cin,
                         int64_t voxels, void* stream);
/* One launch converting four fp32 weights W_i (rows_i, cols_i), row-major, to bf16 in `out` (16-byte aligned): for i = 0..3
 * in turn, W_i as stored with rows ld8(cols_i) elements apart, then W_i^T (cols_i, rows_i) with rows ld8(rows_i) apart,
 * ld8(n) = n rounded up to a multiple of 8, the padding zero.  fz_bf16_staged_elems(rows, cols) is the number of bf16
 * elements one matrix takes (both copies). */
int fz_bf16_stage_weights_supported(int32_t rows, int32_t cols);
int64_t fz_bf16_staged_elems(int32_t rows, int32_t cols);
int fz_bf16_stage_weights(const float* w0, int32_t rows0, int32_t cols0, const float* w1, int32_t rows1, int32_t cols1,
                          const float* w2, int32_t rows2, int32_t cols2, const float* w3, int32_t rows3, int32_t cols3, void* out,
                          void* stream);
/* The same layout for a single weight (the standalone layers): W as stored, then W^T, in one launch. */
int fz_bf16_stage_weight(const float* w, int32_t rows, int32_t cols, void* out, void* stream);
/* fz_layernorm_cf_forward / fz_layernorm_cf_backward_add on bf16 x, y, dy, add, dx; gamma, beta, d(gamma), d(beta) fp32. */
int fz_layernorm_cf_bf16_supported(int32_t channels, int64_t voxels);
int fz_layernorm_cf_forward_bf16(const void* x, const float* gamma, const float* beta, void* y, int64_t batch, int32_t channels,
                                 int64_t voxels, float eps, void* stream);
int fz_layernorm_cf_backward_add_bf16(const void* x, const float* gamma, const void* dy, const void* add, void* dx, float* dgamma,
                                      float* dbeta, int64_t batch, int32_t channels, int64_t voxels, float eps, void* stream);
/* 1 if fz_swnmf_forward / _backward take bf16 volumes of this geometry and solver (g->dtype is ignored). */
int fz_swnmf_bf16_supported(const fz_geom* g, const fz_solver* s, int32_t relu_input);

/* ---- fp16 activations (the FactorizerBlock under fp16 autocast, torch.autocast("cuda")'s default, or fed fp16 tensors) ----
 * The bf16 entry points above with fp16 (torch.float16) in every `void*` buffer: the same kernels, shapes, conditions and
 * FZ_ERR_UNSUPPORTED refusals.  Sums stay fp32 and are rounded to fp16 once (round to nearest even): a result beyond
 * +-65504 becomes +-inf, not a saturated value, so a loss scaler sees the overflow. */
int fz_linear_forward_f16_supported(int32_t cout, int32_t cin, int64_t voxels);
int fz_linear_forward_f16(const void* x, const void* W, int32_t ldw, const float* bias, void* y, int64_t batch, int32_t cin,
                          int32_t cout, int64_t voxels, int32_t epilogue, const void* aux, void* y2, void* stream);
int fz_linear_wgrad_f16_supported(int32_t cout, int32_t cin, int64_t voxels);
int fz_linear_wgrad_f16(const void* dy, const void* x, float* dW, float* db, int64_t batch, int32_t cout, int32_t cin,
                        int64_t voxels, void* stream);
/* fz_bf16_stage_weights' layout (and element counts) with fp16 values. */
int fz_f16_stage_weights_supported(int32_t rows, int32_t cols);
int64_t fz_f16_staged_elems(int32_t rows, int32_t cols);
int fz_f16_stage_weights(const float* w0, int32_t rows0, int32_t cols0, const float* w1, int32_t rows1, int32_t cols1,
                         const float* w2, int32_t rows2, int32_t cols2, const float* w3, int32_t rows3, int32_t cols3, void* out,
                         void* stream);
int fz_f16_stage_weight(const float* w, int32_t rows, int32_t cols, void* out, void* stream);
int fz_layernorm_cf_f16_supported(int32_t channels, int64_t voxels);
int fz_layernorm_cf_forward_f16(const void* x, const float* gamma, const float* beta, void* y, int64_t batch, int32_t channels,
                                int64_t voxels, float eps, void* stream);
int fz_layernorm_cf_backward_add_f16(const void* x, const float* gamma, const void* dy, const void* add, void* dx, float* dgamma,
                                     float* dbeta, int64_t batch, int32_t channels, int64_t voxels, float eps, void* stream);
/* 1 if fz_swnmf_forward / _backward take fp16 volumes of this geometry and solver: the same geometries as bf16. */
int fz_swnmf_f16_supported(const fz_geom* g, const fz_solver* s, int32_t relu_input);

/* (batch, channels, D, H, W) <-> (batch, channels*8, D/2*H/2*W/2) with rows ordered (c, kd, kh, kw): the view on which
 * the reference U-Net's kernel-2 stride-2 down-sampling convolution (factorizer/unet.py:53) and transposed up-sampling
 * convolution (unet.py:97-99) are channel maps.  to_depth != 0: full resolution -> patch rows; 0: the inverse.
 * D, H even and W divisible by 4; in and out 16-byte aligned (FZ_ERR_UNSUPPORTED otherwise). */
int fz_space_depth2_supported(int32_t D, int32_t H, int32_t W);
int fz_space_depth2(const float* in, float* out, int64_t batch, int32_t channels, int32_t D, int32_t H, int32_t W,
                    int32_t to_depth, void* stream);
/* The same permutation of bf16 tensors, with the same conditions. */
int fz_space_depth2_bf16_supported(int32_t D, int32_t H, int32_t W);
int fz_space_depth2_bf16(const void* in, void* out, int64_t batch, int32_t channels, int32_t D, int32_t H, int32_t W,
                         int32_t to_depth, void* stream);

/* 3x3x3 convolution, stride 1, zero padding 1, 1..4 input channels -> 32 output channels: the Swin Factorizer's stem
 * (reference factorizer/factorizer.py:139-140).  x (batch, cin, D, H, W), weight (32, cin, 3, 3, 3), bias 32 floats or
 * NULL, y (batch, 32, D, H, W); fp32 contiguous, W divisible by 4, x and y 16-byte aligned (FZ_ERR_UNSUPPORTED otherwise). */
int fz_conv3d_stem_supported(int32_t cin, int32_t cout, int32_t D, int32_t H, int32_t W);
int fz_conv3d_stem_forward(const float* x, const float* weight, const float* bias, float* y, int64_t batch, int32_t cin,
                           int32_t cout, int32_t D, int32_t H, int32_t W, void* stream);
/* The stem with a bf16 y: x is fp32 or bf16 (x_dtype = FZ_DTYPE_F32 / FZ_DTYPE_BF16), weight and bias fp32, the sums fp32
 * rounded to bf16 once after the bias.  Same conditions as fz_conv3d_stem_forward. */
int fz_conv3d_stem_forward_bf16(const void* x, int32_t x_dtype, const float* weight, const float* bias, void* y, int64_t batch,
                                int32_t cin, int32_t cout, int32_t D, int32_t H, int32_t W, void* stream);
/* The stem's weight gradient on a bf16 dy (batch, 32, D, H, W): dW[o][c][kd][kh][kw] = sum over (batch, voxel v) of
 * dy[o][v] x[c][v + (kd-1, kh-1, kw-1)] (zero outside the volume) and db[o] = sum of dy[o][v] (db may be NULL), fp32,
 * OVERWRITTEN.  x is fp32 (read as bf16) or bf16.  tcgen05 kind::f16 on im2col rows built in shared memory, never in
 * global memory.  1..4 -> 32 channels, W divisible by 8, dy and x 16-byte aligned (FZ_ERR_UNSUPPORTED otherwise). */
int fz_conv3d_stem_wgrad_bf16_supported(int32_t cin, int32_t cout, int32_t D, int32_t H, int32_t W);
int fz_conv3d_stem_wgrad_bf16(const void* dy, const void* x, int32_t x_dtype, float* dW, float* db, int64_t batch, int32_t cin,
                              int32_t cout, int32_t D, int32_t H, int32_t W, void* stream);

/* ---- FactMixer / FactorizerBlock pointwise glue, 32-channel blocks (SURVEY section 8(f) row 1) --------
 * All tensors are (batch, channels, voxels) fp32 = flattened NCDHW; weights are the reference's Conv1d(k=1)
 * weights squeezed to (out, in) (factorizer/layers/linear.py:43-50).  Gradient outputs are OVERWRITTEN. */

/* 1 if the four kernels below handle this block: 32 channels, an even number of voxels, MLP hidden width a
 * multiple of 8 up to 256 (the backward runs in slices of 64 hidden units). */
int fz_glue_supported(int32_t channels, int32_t hidden, int64_t voxels);

/* Which glue kernels run on the tensor cores (tcgen05 / TMEM, 3xTF32), for calls made by the CALLING THREAD: bit 0 =
 * fz_ln_linear_forward and fz_mixer_mlp_forward (hidden width 32 or 64), bit 1 = fz_linear_backward, bit 2 =
 * fz_mlp_backward (hidden width 64).  Default 7 = all; 0 = the FP32-pipe kernels.  Both families meet the same parity
 * bounds; the switch exists for the parity tests and for timing one against the other.  No environment variable, no
 * process-wide state. */
void fz_set_glue_mode(int32_t mode);
int fz_get_glue_mode(void);

/* z = W LN(x): norm1 + bias-free in_proj (factorizer/factorizer.py:26,38,75; layers/norm.py:29-34). */
int fz_ln_linear_forward(const float* x, const float* gamma, const float* beta, const float* W, float* z, int64_t batch,
                         int32_t channels, int64_t voxels, float eps, void* stream);

/* x1 = x + W_out m + b_out ; out = x1 + W2 gelu(W1 LN(x1) + b1) + b2: out_proj + residual
 * (factorizer.py:53,75) and norm2 + MLP + residual (factorizer.py:76, layers/mlp.py:54-60, exact-erf GELU).
 * x1 may be NULL (inference); the backward needs it. */
int fz_mixer_mlp_forward(const float* x, const float* m, const float* Wout, const float* bout, const float* gamma,
                         const float* beta, const float* W1, const float* b1, const float* W2, const float* b2, float* x1,
                         float* out, int64_t batch, int32_t channels, int32_t hidden, int64_t voxels, float eps, void* stream);

/* Backward of out = x1 + MLP(LN(x1)): dx1 and the gradients of gamma/beta (LN), W1 (hidden,channels), b1, W2
 * (channels,hidden), b2.  Replaces autograd's replay of layers/mlp.py:54-60 + layers/norm.py:29-34. */
int fz_mlp_backward(const float* x1, const float* dout, const float* gamma, const float* beta, const float* W1,
                    const float* b1, const float* W2, float* dx1, float* dgamma, float* dbeta, float* dW1, float* db1,
                    float* dW2, float* db2, int64_t batch, int32_t channels, int32_t hidden, int64_t voxels, float eps,
                    void* stream);

/* Backward of y = W n(a) (+ b) with n = LayerNorm (layernorm != 0) or identity:
 *   da = W^T dy, through the LayerNorm when there is one, plus `resid` (the gradient arriving over the residual
 *   connection; may be NULL); dW = sum dy n(a)^T; db = sum dy (may be NULL); d(gamma), d(beta) (LayerNorm only).
 * Serves out_proj (a = m, no LayerNorm) and in_proj + norm1 (a = x, resid = dx1). */
int fz_linear_backward(const float* dy, const float* a, const float* gamma, const float* beta, const float* W,
                       const float* resid, float* da, float* dW, float* db, float* dgamma, float* dbeta, int64_t batch,
                       int32_t channels, int64_t voxels, float eps, int32_t layernorm, void* stream);

/* Which implementation the last fz_swnmf_* call on this thread used: 0 = generic shared-memory
 * kernels, 1 = the window-at-a-time TMA/register kernels (8x512 windows, rank-1 HALS, any shifts),
 * 2 = the three-pass octant kernels (the same with shifts [0, patch/2] and ReLU: the default
 * Swin-Factorizer block), 3 = the sub-warp-per-matrix register kernels for small matrices (64 columns with
 * 4..32 rows, 8x16, 8x128, 8x256; rank-1 HALS / MU, at most 5 sweeps; also used by fz_nmf_* when only y / dy
 * are involved), 4 = the octant kernels once per pair of window sets (a, a + patch/2) on the volume rolled by a
 * (e.g. shifts [0, 2, 4, 6]), 5 = one grid-wide pass per sweep for a single huge matrix per (sample, head)
 * (Matricize(grid_size=1), rank-1 MU / HALS), 6 = the octant kernels as one persistent, software-pipelined launch per
 * direction (volumes beyond the L2).  For tests and the benchmark's bookkeeping. */
int fz_last_path(void);
/* Number of kernel launches issued by the last fz_* call on this thread. */
int fz_last_launches(void);
#ifdef __cplusplus
}
#endif
#endif /* FACTORIZER_B200_H_ */
