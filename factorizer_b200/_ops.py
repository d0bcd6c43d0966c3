"""torch.autograd.Function wrappers over the C ABI.  PyTorch provides device memory, streams and
autograd bookkeeping; every byte of arithmetic happens in libfactorizer_b200.so."""
from __future__ import annotations

import ctypes
import threading
from typing import Optional, Sequence, Tuple

import torch
from torch.autograd.function import once_differentiable

from . import _lib as L


class Geometry:
    """Window geometry of a (SW)Matricize for a given input (hashable, batch-independent)."""

    def __init__(self, channels: int, size: Sequence[int], patch: Sequence[int], head_dim: int,
                 shifts: Sequence[Sequence[int]]):
        self.channels = int(channels)
        self.size = tuple(int(s) for s in size)
        self.patch = tuple(int(p) for p in patch)
        self.head_dim = int(head_dim)
        self.shifts = tuple(tuple(int(v) for v in s) for s in shifts)
        self.path = L.FZ_PATH_AUTO       # fz_geom.path: restrict the kernel family (tests / measurements)
        self.heads = self.channels // self.head_dim
        self.grid = tuple(s // p for s, p in zip(self.size, self.patch))
        self.num_windows = 1
        self.num_cols = 1
        for g, p in zip(self.grid, self.patch):
            self.num_windows *= g
            self.num_cols *= p

    def c_geom(self, batch: int, dtype: torch.dtype = torch.float32) -> L.FzGeom:
        return L.make_geom(batch, self.channels, self.size, self.patch, self.head_dim, self.shifts, self.path,
                           {torch.bfloat16: L.FZ_DTYPE_BF16, torch.float16: L.FZ_DTYPE_F16}.get(dtype, L.FZ_DTYPE_F32))

    def mat_shape(self, batch: int) -> Tuple[int, int, int, int]:
        return (len(self.shifts) * batch * self.heads, self.num_windows, self.head_dim, self.num_cols)

    def vol_shape(self, batch: int) -> Tuple[int, ...]:
        return (batch, self.channels, *self.size)


class SolverSpec:
    def __init__(self, kind: int, rank: int, num_iters: int, num_grad_steps: int, eps: float = 1e-16):
        self.kind, self.rank, self.num_iters = int(kind), int(rank), int(num_iters)
        self.num_grad_steps, self.eps = int(num_grad_steps), float(eps)

    def c_solver(self) -> L.FzSolver:
        return L.make_solver(self.kind, self.rank, self.num_iters, self.num_grad_steps, self.eps)


class _GradModeFunction(torch.autograd.Function):
    """autograd.Function whose forward can tell whether a backward may follow.  Function.forward always runs with grad
    mode off and ctx.needs_input_grad only reflects requires_grad of the inputs, so under torch.no_grad() (inference
    with an unfrozen model) it would still ask for the saved buffers; the caller's grad mode is recorded on entry."""
    _caller = threading.local()

    @classmethod
    def apply(cls, *args, **kwargs):
        _GradModeFunction._caller.grad = torch.is_grad_enabled()
        return super().apply(*args, **kwargs)

    @staticmethod
    def wants_grad(ctx, upto=None) -> bool:
        flags = ctx.needs_input_grad if upto is None else ctx.needs_input_grad[:upto]
        return bool(getattr(_GradModeFunction._caller, "grad", True)) and any(flags)


def _check_vol(x: torch.Tensor, geom: Geometry, name: str, allow_16bit: bool = False) -> torch.Tensor:
    x = L.require_cuda_f32(x, name, allow_bf16=allow_16bit, allow_f16=allow_16bit)
    if tuple(x.shape[1:]) != (geom.channels, *geom.size):
        raise ValueError(f"{name}: expected (B, {geom.channels}, {', '.join(map(str, geom.size))}), "
                         f"got {tuple(x.shape)}")
    return x


def _check_mat(y: torch.Tensor, geom: Geometry, name: str) -> Tuple[torch.Tensor, int]:
    y = L.require_cuda_f32(y, name)
    S = len(geom.shifts)
    if y.dim() != 4 or tuple(y.shape[1:]) != (geom.num_windows, geom.head_dim, geom.num_cols) \
            or y.shape[0] % (S * geom.heads):
        raise ValueError(f"{name}: expected (S*B*{geom.heads}, {geom.num_windows}, {geom.head_dim}, "
                         f"{geom.num_cols}), got {tuple(y.shape)}")
    return y, y.shape[0] // (S * geom.heads)


class LaunchCounter:
    """Kernel launches issued through this module (every C entry point reports its own count, read here on the calling
    thread -- autograd runs backward on its own).  bench.py reads it for `gpu_launches`."""
    _lock = threading.Lock()
    total = 0

    @classmethod
    def add(cls, n: int) -> None:
        with cls._lock:
            cls.total += n


def _call(fn, *args) -> None:
    L.check(fn(*args))
    LaunchCounter.add(L.lib().fz_last_launches())


# ---- standalone matricize ------------------------------------------------------------------------
def _gather(x, geom: Geometry, divide: bool):
    lib = L.lib()
    B = x.shape[0]
    y = torch.empty(geom.mat_shape(B), device=x.device, dtype=torch.float32)
    g = geom.c_geom(B)
    with torch.cuda.device(x.device):
        fn = lib.fz_swmat_inverse_adjoint if divide else lib.fz_swmat_forward
        _call(fn, L.ptr(x), L.ptr(y), ctypes.byref(g), L.stream_ptr(x.device))
    return y


def _scatter(y, batch: int, geom: Geometry, reference_inverse: bool):
    lib = L.lib()
    out = torch.empty(geom.vol_shape(batch), device=y.device, dtype=torch.float32)
    g = geom.c_geom(batch)
    with torch.cuda.device(y.device):
        fn = lib.fz_swmat_inverse if reference_inverse else lib.fz_swmat_forward_adjoint
        _call(fn, L.ptr(y), L.ptr(out), ctypes.byref(g), L.stream_ptr(y.device))
    return out


class SWMatForward(torch.autograd.Function):
    """SWMatricize.forward / Matricize.forward (reference operations.py:266-272, 417-421)."""

    @staticmethod
    def forward(ctx, x, geom: Geometry):
        x = _check_vol(x, geom, "x")
        ctx.geom = geom
        ctx.batch = x.shape[0]
        return _gather(x, geom, divide=False)

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        gy, _ = _check_mat(gy, ctx.geom, "grad")
        return _scatter(gy, ctx.batch, ctx.geom, reference_inverse=False), None


class SWMatInverse(torch.autograd.Function):
    """SWMatricize.inverse_forward (operations.py:423-434) when ``averaged``; the plain
    Reshape.inverse_forward (operations.py:274-280) otherwise."""

    @staticmethod
    def forward(ctx, y, geom: Geometry, averaged: bool):
        y, batch = _check_mat(y, geom, "y")
        ctx.geom, ctx.averaged = geom, averaged
        return _scatter(y, batch, geom, reference_inverse=averaged)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        g = _check_vol(g, ctx.geom, "grad")
        return _gather(g, ctx.geom, divide=ctx.averaged), None, None


# ---- NMF on matricised tensors -------------------------------------------------------------------
def _nmf_forward(x3, u0, v0, spec: SolverSpec, want_uv: bool, want_y: bool):
    lib = L.lib()
    n, M, N = x3.shape
    R = spec.rank
    u = torch.empty((n, M, R), device=x3.device, dtype=torch.float32) if want_uv else None
    v = torch.empty((n, N, R), device=x3.device, dtype=torch.float32) if want_uv else None
    y = torch.empty((n, M, N), device=x3.device, dtype=torch.float32) if want_y else None
    s = spec.c_solver()
    if n == 0:
        return u, v, y
    with torch.cuda.device(x3.device):
        _call(lib.fz_nmf_forward, L.ptr(x3), L.ptr(u0), L.ptr(v0), L.ptr(u), L.ptr(v), L.ptr(y), n, M, N,
              ctypes.byref(s), L.stream_ptr(x3.device))
    return u, v, y


def _nmf_backward(x3, u0, v0, gy, gu, gv, spec: SolverSpec):
    lib = L.lib()
    n, M, N = x3.shape
    gx = torch.empty_like(x3)
    s = spec.c_solver()
    if n == 0:
        return gx
    with torch.cuda.device(x3.device):
        _call(lib.fz_nmf_backward, L.ptr(x3), L.ptr(u0), L.ptr(v0), L.ptr(gy), L.ptr(gu), L.ptr(gv),
              L.ptr(gx), n, M, N, ctypes.byref(s), L.stream_ptr(x3.device))
    return gx


def _flatten_batch(x: torch.Tensor, size) -> torch.Tensor:
    M, N = size
    if x.dim() < 2 or tuple(x.shape[-2:]) != (M, N):
        raise ValueError(f"NMF built for matrices of size {(M, N)}, got input of shape {tuple(x.shape)}")
    return x.reshape(-1, M, N)


# a rank-1 matrix this large has no single-CTA kernel: it runs as the one-window-per-sample case of the fused core
# (csrc/fz_nmf_big.cu), whose entry points carry the scratch buffers the grid-wide passes need
_BIG_ELEMS = 16384


def _as_one_window_volume(spec: SolverSpec, size):
    M, N = size
    if spec.rank != 1 or M * N < _BIG_ELEMS:
        return None
    return Geometry(channels=M, size=(N,), patch=(N,), head_dim=M, shifts=[(0,)])


class NMFReconstruct(_GradModeFunction):
    """MatrixFactorization.forward = reconstruct(decompose(x))
    (reference matrix_factorization.py:514-533, 544-546) as one kernel per direction."""

    @staticmethod
    def forward(ctx, x, u0, v0, spec: SolverSpec, size):
        x = L.require_cuda_f32(x, "x")
        x3 = _flatten_batch(x, size)
        u0 = L.require_cuda_f32(u0, "u0")
        v0 = L.require_cuda_f32(v0, "v0")
        geom = _as_one_window_volume(spec, size) if x3.shape[0] > 0 else None
        saved = None
        if geom is not None:
            y, saved = _swnmf_forward(x3, u0, v0, geom, spec, False, _GradModeFunction.wants_grad(ctx, 1))
        else:
            _, _, y = _nmf_forward(x3, u0, v0, spec, want_uv=False, want_y=True)
        ctx.save_for_backward(x3, u0, v0, saved)
        ctx.spec, ctx.shape, ctx.geom = spec, x.shape, geom
        return y.reshape(x.shape)

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        x3, u0, v0, saved = ctx.saved_tensors
        gy = L.require_cuda_f32(gy, "grad").reshape(x3.shape)
        if ctx.geom is not None:
            gx = _swnmf_backward(x3, gy, u0, v0, saved, ctx.geom, ctx.spec, False)
        else:
            gx = _nmf_backward(x3, u0, v0, gy, None, None, ctx.spec)
        return gx.reshape(ctx.shape), None, None, None, None


class NMFDecompose(torch.autograd.Function):
    """MatrixFactorization.decompose (matrix_factorization.py:514-530): returns (u, v)."""

    @staticmethod
    def forward(ctx, x, u0, v0, spec: SolverSpec, size):
        x = L.require_cuda_f32(x, "x")
        x3 = _flatten_batch(x, size)
        u0 = L.require_cuda_f32(u0, "u0")
        v0 = L.require_cuda_f32(v0, "v0")
        u, v, _ = _nmf_forward(x3, u0, v0, spec, want_uv=True, want_y=False)
        ctx.save_for_backward(x3, u0, v0)
        ctx.spec, ctx.shape = spec, x.shape
        batch = x.shape[:-2]
        return u.reshape(*batch, size[0], spec.rank), v.reshape(*batch, size[1], spec.rank)

    @staticmethod
    @once_differentiable
    def backward(ctx, gu, gv):
        x3, u0, v0 = ctx.saved_tensors
        n, M, N = x3.shape
        R = ctx.spec.rank
        gu = None if gu is None else L.require_cuda_f32(gu, "grad_u").reshape(n, M, R)
        gv = None if gv is None else L.require_cuda_f32(gv, "grad_v").reshape(n, N, R)
        gx = _nmf_backward(x3, u0, v0, None, gu, gv, ctx.spec)
        return gx.reshape(ctx.shape), None, None, None, None


# ---- fused FactMixer core ------------------------------------------------------------------------
_workspaces = {}


def _workspace(device, nbytes: int) -> Optional[torch.Tensor]:
    """Per-(device, stream) scratch for the tile-order counters; grown on demand, never shrunk."""
    if nbytes == 0:
        return None
    key = (device, torch.cuda.current_stream(device).cuda_stream)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.zeros(nbytes, device=device, dtype=torch.uint8)
        _workspaces[key] = ws
    return ws


def _swnmf_forward(x, u0, v0, geom: Geometry, spec: SolverSpec, relu: bool, need_grad: bool):
    """One launch sequence of the fused core; returns (y, saved-for-backward buffer or None)."""
    lib = L.lib()
    g, s = geom.c_geom(x.shape[0], x.dtype), spec.c_solver()
    y = torch.empty_like(x)
    saved = None
    with torch.cuda.device(x.device):
        nsaved = lib.fz_swnmf_saved_bytes(ctypes.byref(g), ctypes.byref(s)) if need_grad else 0
        if nsaved:
            saved = torch.empty(nsaved, device=x.device, dtype=torch.uint8)
        ws = _workspace(x.device, lib.fz_swnmf_workspace_bytes(ctypes.byref(g), ctypes.byref(s)))
        _call(lib.fz_swnmf_forward, L.ptr(x), L.ptr(u0), L.ptr(v0), L.ptr(y), L.ptr(saved), L.ptr(ws),
              ctypes.byref(g), ctypes.byref(s), int(relu), L.stream_ptr(x.device))
    return y, saved


def _swnmf_backward(x, gy, u0, v0, saved, geom: Geometry, spec: SolverSpec, relu: bool):
    lib = L.lib()
    g, s = geom.c_geom(x.shape[0], x.dtype), spec.c_solver()
    gx = torch.empty_like(x)
    with torch.cuda.device(x.device):
        ws = _workspace(x.device, lib.fz_swnmf_workspace_bytes(ctypes.byref(g), ctypes.byref(s)))
        _call(lib.fz_swnmf_backward, L.ptr(x), L.ptr(gy), L.ptr(u0), L.ptr(v0), L.ptr(saved), L.ptr(gx),
              L.ptr(ws), ctypes.byref(g), ctypes.byref(s), int(relu), L.stream_ptr(x.device))
    return gx


class SWNMF(_GradModeFunction):
    """reshape -> act -> factorize -> reshape.inverse_forward of FactMixer.forward
    (reference factorizer/factorizer.py:41-50): X is read once and Y written once."""

    @staticmethod
    def forward(ctx, x, u0, v0, geom: Geometry, spec: SolverSpec, relu: bool):
        # bf16 and fp16 volumes (an extension: the reference runs fp32) are read and written in their type by the octant and
        # sub-warp kernels; u0, v0, the saved records and all arithmetic stay fp32
        x = _check_vol(x, geom, "x", allow_16bit=True)
        u0 = L.require_cuda_f32(u0.float(), "u0")
        v0 = L.require_cuda_f32(v0.float(), "v0")
        y, saved = _swnmf_forward(x, u0, v0, geom, spec, relu, _GradModeFunction.wants_grad(ctx, 1))
        ctx.save_for_backward(x, u0, v0, saved)
        ctx.geom, ctx.spec, ctx.relu = geom, spec, relu
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        x, u0, v0, saved = ctx.saved_tensors
        gy = _check_vol(gy.to(x.dtype), ctx.geom, "grad", allow_16bit=True)
        gx = _swnmf_backward(x, gy, u0, v0, saved, ctx.geom, ctx.spec, ctx.relu)
        return gx, None, None, None, None, None


# ---- whole FactorizerBlock: fused glue kernels around the fused core --------------------------------
def block_glue_supported(x: torch.Tensor, hidden: int) -> bool:
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() >= 3):
        return False
    vox = 1
    for s in x.shape[2:]:
        vox *= s
    return bool(L.lib().fz_glue_supported(x.shape[1], int(hidden), vox))


class FactorizerBlockFn(_GradModeFunction):
    """FactorizerBlock.forward (reference factorizer/factorizer.py:74-77 with FactMixer.forward :34-57) for
    norm = LayerNorm, act = ReLU, no dropout: three launches forward (norm1+in_proj | fused matricize+NMF core |
    out_proj+residual+norm2+MLP+residual), four backward.  Saves x, z (in_proj output), m (core output) and x1
    (after the first residual); every intermediate of the MLP is recomputed in the backward kernel."""

    @staticmethod
    def forward(ctx, x, g1, b1n, w_in, w_out, b_out, g2, b2n, w1, bb1, w2, bb2, u0, v0, geom, spec, eps1, eps2):
        lib = L.lib()
        x = _check_vol(x, geom, "x")
        params = [L.require_cuda_f32(t, "parameter") for t in (g1, b1n, w_in, w_out, b_out, g2, b2n, w1, bb1, w2, bb2)]
        g1, b1n, w_in, w_out, b_out, g2, b2n, w1, bb1, w2, bb2 = params
        u0 = L.require_cuda_f32(u0, "u0")
        v0 = L.require_cuda_f32(v0, "v0")
        B, C = x.shape[0], x.shape[1]
        vox = x.numel() // max(B * C, 1)
        hid = w1.shape[0]
        need_grad = _GradModeFunction.wants_grad(ctx, 12)
        st = L.stream_ptr(x.device)
        z = torch.empty_like(x)
        out = torch.empty_like(x)
        x1 = torch.empty_like(x) if need_grad else None
        with torch.cuda.device(x.device):
            _call(lib.fz_ln_linear_forward, L.ptr(x), L.ptr(g1), L.ptr(b1n), L.ptr(w_in), L.ptr(z), B, C, vox, float(eps1), st)
            m, saved = _swnmf_forward(z, u0, v0, geom, spec, True, need_grad)
            _call(lib.fz_mixer_mlp_forward, L.ptr(x), L.ptr(m), L.ptr(w_out), L.ptr(b_out), L.ptr(g2), L.ptr(b2n),
                  L.ptr(w1), L.ptr(bb1), L.ptr(w2), L.ptr(bb2), L.ptr(x1), L.ptr(out), B, C, hid, vox, float(eps2), st)
        if need_grad:
            ctx.save_for_backward(x, z, m, x1, saved, g1, b1n, w_in, w_out, g2, b2n, w1, bb1, w2, u0, v0)
            ctx.geom, ctx.spec, ctx.eps = geom, spec, (float(eps1), float(eps2))
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, gout):
        lib = L.lib()
        x, z, m, x1, saved, g1, b1n, w_in, w_out, g2, b2n, w1, bb1, w2, u0, v0 = ctx.saved_tensors
        gout = _check_vol(gout, ctx.geom, "grad")
        B, C = x.shape[0], x.shape[1]
        vox = x.numel() // max(B * C, 1)
        hid = w1.shape[0]
        eps1, eps2 = ctx.eps
        st = L.stream_ptr(x.device)
        new = lambda t: torch.empty_like(t)
        dg2, db2n, dw1, dbb1, dw2, dbb2 = new(g2), new(b2n), new(w1), new(bb1), new(w2), torch.empty(C, device=x.device)
        dw_out, db_out, dw_in, dg1, db1n = new(w_out), torch.empty(C, device=x.device), new(w_in), new(g1), new(b1n)
        dx1 = torch.empty_like(x)
        with torch.cuda.device(x.device):
            _call(lib.fz_mlp_backward, L.ptr(x1), L.ptr(gout), L.ptr(g2), L.ptr(b2n), L.ptr(w1), L.ptr(bb1), L.ptr(w2),
                  L.ptr(dx1), L.ptr(dg2), L.ptr(db2n), L.ptr(dw1), L.ptr(dbb1), L.ptr(dw2), L.ptr(dbb2), B, C, hid, vox,
                  eps2, st)
            dm = torch.empty_like(x)
            _call(lib.fz_linear_backward, L.ptr(dx1), L.ptr(m), None, None, L.ptr(w_out), None, L.ptr(dm),
                  L.ptr(dw_out), L.ptr(db_out), None, None, B, C, vox, 0.0, 0, st)
            dz = _swnmf_backward(z, dm, u0, v0, saved, ctx.geom, ctx.spec, True)
            dx = dm                         # dm is dead once the core's backward has run: reuse its storage
            _call(lib.fz_linear_backward, L.ptr(dz), L.ptr(x), L.ptr(g1), L.ptr(b1n), L.ptr(w_in), L.ptr(dx1), L.ptr(dx),
                  L.ptr(dw_in), None, L.ptr(dg1), L.ptr(db1n), B, C, vox, eps1, 1, st)
        return (dx, dg1, db1n, dw_in, dw_out, db_out, dg2, db2n, dw1, dbb1, dw2, dbb2,
                None, None, None, None, None, None)


# ---- FactorizerBlock of any width: channel-map kernels with fused epilogues around the fused core ------------------
EPI_NONE, EPI_RESIDUAL, EPI_GELU, EPI_GELU_GRAD, EPI_GELU_ONLY = 0, 1, 2, 3, 4


def _channel_map(x, w, bias, epi=EPI_NONE, aux=None, transposed=False):
    """r = W x + bias on (B, C_in, voxels) with the epilogues of fz_linear_forward_ex (csrc/fz_linear_tc.cu); returns y,
    or (y, gelu(y)) for EPI_GELU.  transposed: w is the (C_in, C_out) matrix of the layer whose input gradient this is,
    read as it lies.  Shapes the kernel does not take (unaligned views) run the same arithmetic in torch."""
    lib = L.lib()
    B, cin, vox = x.shape
    w = w.contiguous()
    cout = w.shape[1] if transposed else w.shape[0]
    if (x.is_contiguous() and lib.fz_linear_forward_supported(cout, cin, vox) and (x.data_ptr() | w.data_ptr()) % 16 == 0
            and (aux is None or aux.is_contiguous()) and not (transposed and cout % 4)):
        y = torch.empty(B, cout, vox, device=x.device, dtype=torch.float32)
        y2 = torch.empty_like(y) if epi == EPI_GELU else None
        _call(lib.fz_linear_forward_ex, L.ptr(x), L.ptr(w), L.ptr(bias), L.ptr(y), B, cin, cout, vox, epi, int(transposed),
              L.ptr(aux), L.ptr(y2), L.stream_ptr(x.device))
        return (y, y2) if epi == EPI_GELU else y
    wb = (w.t() if transposed else w).unsqueeze(0).expand(B, -1, -1)
    r = torch.bmm(wb, x) if bias is None else torch.baddbmm(bias[None, :, None], wb, x)
    if epi == EPI_RESIDUAL:
        return r + aux
    if epi == EPI_GELU:
        return r, torch.nn.functional.gelu(r)
    if epi == EPI_GELU_GRAD:
        return torch.ops.aten.gelu_backward(r, aux)
    if epi == EPI_GELU_ONLY:
        return torch.nn.functional.gelu(r)
    return r


# the suffix of the C entry points of each 16-bit activation type (fz_linear_forward_bf16 / _f16, fz_bf16_stage_weights /
# fz_f16_stage_weights, ...)
_HALF = {torch.bfloat16: "bf16", torch.float16: "f16"}


def _channel_map_wgrad(gy, x, want_bias: bool):
    """dW = sum over (batch, voxels) of gy x^T, db = sum of gy, both fp32.  bf16 / fp16 gy and x: fz_linear_wgrad_bf16 / _f16.
    fp32 views the kernels do not take (non-contiguous, or not 16-byte aligned) run the same arithmetic in torch."""
    lib = L.lib()
    B, cout, vox = gy.shape
    cin = x.shape[1]
    half = _HALF.get(x.dtype)
    if half or (gy.is_contiguous() and x.is_contiguous() and (gy.data_ptr() | x.data_ptr()) % 16 == 0
                and lib.fz_linear_wgrad_supported(cout, cin, vox)):
        gw = torch.empty(cout, cin, device=x.device, dtype=torch.float32)
        gb = torch.empty(cout, device=x.device, dtype=torch.float32) if want_bias else None
        fn = getattr(lib, f"fz_linear_wgrad_{half}") if half else lib.fz_linear_wgrad
        _call(fn, L.ptr(gy), L.ptr(x), L.ptr(gw), L.ptr(gb), B, cout, cin, vox, L.stream_ptr(x.device))
        return gw, gb
    gw = torch.bmm(gy, x.transpose(1, 2)).sum(0)
    return gw, (gy.sum((0, 2)) if want_bias else None)


def _ln_forward(x3, gamma, beta, eps):
    """LayerNorm over the channels of fp32, bf16 or fp16 (B, C, voxels); the statistics are fp32."""
    lib = L.lib()
    B, C, vox = x3.shape
    y = torch.empty_like(x3)
    half = _HALF.get(x3.dtype)
    fn = getattr(lib, f"fz_layernorm_cf_forward_{half}") if half else lib.fz_layernorm_cf_forward
    _call(fn, L.ptr(x3), L.ptr(gamma), L.ptr(beta), L.ptr(y), B, C, vox, float(eps), L.stream_ptr(x3.device))
    return y


def _ln_backward_add(x3, gamma, gy, add, eps):
    """dx = add + LN'(gy) in the dtype of x3, d(gamma), d(beta) in fp32."""
    lib = L.lib()
    B, C, vox = x3.shape
    dx, dg, db = torch.empty_like(x3), torch.empty_like(gamma), torch.empty_like(gamma)
    half = _HALF.get(x3.dtype)
    fn = getattr(lib, f"fz_layernorm_cf_backward_add_{half}") if half else lib.fz_layernorm_cf_backward_add
    _call(fn, L.ptr(x3), L.ptr(gamma), L.ptr(gy), L.ptr(add), L.ptr(dx), L.ptr(dg), L.ptr(db), B, C, vox, float(eps),
          L.stream_ptr(x3.device))
    return dx, dg, db


def wide_block_supported(x: torch.Tensor, hidden: int) -> bool:
    """FactorizerBlockWideFn: any channel count the channel-map and LayerNorm kernels take (multiples of 4 up to 512),
    voxel counts that are multiples of 4, fp32, no autocast."""
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() >= 3 and x.is_contiguous()):
        return False
    if torch.is_autocast_enabled():
        return False
    B, C = x.shape[0], x.shape[1]
    vox = x.numel() // max(B * C, 1)
    lib = L.lib()
    return bool(B > 0 and vox > 0 and lib.fz_layernorm_cf_supported(C, vox) and lib.fz_linear_forward_supported(C, C, vox)
                and lib.fz_linear_forward_supported(int(hidden), C, vox) and lib.fz_linear_forward_supported(C, int(hidden), vox)
                and x.data_ptr() % 16 == 0)


class _WideBlockFn(_GradModeFunction):
    """FactorizerBlock.forward (reference factorizer/factorizer.py:74-77 with FactMixer.forward :34-57, MLP
    layers/mlp.py:54-60) for norm = LayerNorm, act = ReLU, GELU MLP, no dropout, at any width: every step is a kernel of this
    library, with the residual sums, the bias + GELU and the GELU derivative folded into the epilogues of the tensor-core
    channel map and the residual gradients into the LayerNorm backward -- nine launches forward (norm1 | in_proj | core x3 |
    out_proj + residual | norm2 | fc1 + GELU | fc2 + residual), the same steps in reverse backward.  Written once for
    FactorizerBlockWideFn, FactorizerBlockBf16Fn and FactorizerBlockF16Fn; a subclass names the activations' `dtype` and says how its channel maps
    read the four weights (w_in, w_out, w1, w2): _stage(ws) returns the tensors the backward keeps for them, _maps(staged,
    shapes) one channel map per weight, m(x, bias, epi, aux, transposed), transposed = that layer's input gradient."""
    dtype = None

    @classmethod
    def _forward(cls, ctx, x, g1, b1n, w_in, w_out, b_out, g2, b2n, w1, bb1, w2, bb2, u0, v0, geom, spec, eps1, eps2):
        if x.dtype != cls.dtype:
            raise NotImplementedError(f"factorizer_b200: {cls.__name__} takes {cls.dtype} activations, got {x.dtype}")
        x = _check_vol(x, geom, "x", allow_16bit=True)
        params = [L.require_cuda_f32(t, "parameter") for t in (g1, b1n, w_in, w_out, b_out, g2, b2n, w1, bb1, w2, bb2)]
        g1, b1n, w_in, w_out, b_out, g2, b2n, w1, bb1, w2, bb2 = params
        u0 = L.require_cuda_f32(u0, "u0")
        v0 = L.require_cuda_f32(v0, "v0")
        B, C = x.shape[0], x.shape[1]
        need_grad = _GradModeFunction.wants_grad(ctx, 12)
        x3 = x.view(B, C, -1)
        shapes = [tuple(w.shape) for w in (w_in, w_out, w1, w2)]
        with torch.cuda.device(x.device):
            staged = cls._stage((w_in, w_out, w1, w2))
            m_in, m_out, m1, m2 = cls._maps(staged, shapes)
            n1 = _ln_forward(x3, g1, b1n, eps1)
            z = m_in(n1, None)
            m, saved = _swnmf_forward(z.view(x.shape), u0, v0, geom, spec, True, need_grad)
            m3 = m.view(B, C, -1)
            x1 = m_out(m3, b_out, EPI_RESIDUAL, x3)
            n2 = _ln_forward(x1, g2, b2n, eps2)
            if need_grad:
                h, g = m1(n2, bb1, EPI_GELU)
            else:                                                       # inference: the pre-activation is not kept
                h, g = None, m1(n2, bb1, EPI_GELU_ONLY)
            out = m2(g, bb2, EPI_RESIDUAL, x1)
        if need_grad:
            ctx.save_for_backward(x3, n1, z, m3, x1, n2, h, g, saved, g1, g2, u0, v0, *staged)
            ctx.block, ctx.shapes = cls, shapes
            ctx.geom, ctx.spec, ctx.eps = geom, spec, (float(eps1), float(eps2))
        return out.view(x.shape)

    @staticmethod
    @once_differentiable
    def backward(ctx, gout):
        x3, n1, z, m3, x1, n2, h, g, saved, g1, g2, u0, v0, *staged = ctx.saved_tensors
        geom = ctx.geom
        gout = _check_vol(gout.to(x3.dtype), geom, "grad", allow_16bit=True)
        B, C = x3.shape[0], x3.shape[1]
        eps1, eps2 = ctx.eps
        m_in, m_out, m1, m2 = ctx.block._maps(staged, ctx.shapes)
        go3 = gout.view(B, C, -1)
        with torch.cuda.device(x3.device):
            dh = m2(go3, None, EPI_GELU_GRAD, h, True)                      # (W2^T dOut) * gelu'(h)
            dw2, dbb2 = _channel_map_wgrad(go3, g, True)
            dw1, dbb1 = _channel_map_wgrad(dh, n2, True)
            dn2 = m1(dh, None, transposed=True)
            dx1, dg2, db2n = _ln_backward_add(x1, g2, dn2, go3, eps2)       # dOut + norm2'(..)
            dm = m_out(dx1, None, transposed=True)
            dw_out, db_out = _channel_map_wgrad(dx1, m3, True)
            vol = (B, C, *geom.size)
            dz = _swnmf_backward(z.view(vol), dm.view(vol), u0, v0, saved, geom, ctx.spec, True).view(B, C, -1)
            dw_in, _ = _channel_map_wgrad(dz, n1, False)
            dn1 = m_in(dz, None, transposed=True)
            dx, dg1, db1n = _ln_backward_add(x3, g1, dn1, dx1, eps1)        # dx1 + norm1'(..)
        return (dx.view(vol), dg1, db1n, dw_in, dw_out, db_out, dg2, db2n, dw1, dbb1, dw2, dbb2,
                None, None, None, None, None, None)


class FactorizerBlockWideFn(_WideBlockFn):
    """_WideBlockFn on fp32 activations (the 64..512-channel stages of the Swin Factorizer): the tcgen05 channel map
    (fz_linear_forward_ex, 3xTF32) reads the four weights as stored, and transposed in place for the input gradients."""
    dtype = torch.float32

    @staticmethod
    def forward(ctx, *args):
        return FactorizerBlockWideFn._forward(ctx, *args)

    @staticmethod
    def _stage(ws):
        return ws

    @staticmethod
    def _maps(ws, shapes):
        def bind(w):
            return lambda x, bias, epi=EPI_NONE, aux=None, transposed=False: _channel_map(x, w, bias, epi, aux, transposed)
        return [bind(w) for w in ws]


# ---- FactorizerBlock on bf16 activations: bf16 tensor-core channel maps around the bf16 fused core ------------------
def _ld8(n: int) -> int:
    return (int(n) + 7) & ~7


def bf16_core_supported(geom: Geometry, spec: SolverSpec, relu: bool = True) -> bool:
    """The fused core takes bf16 volumes of this geometry: the octant kernels (head_dim 8, patch 8^3, rank-1 HALS, an even
    number of patches along W) at shifts [0, 4], or at window sets that pair up as (a, a + 4) with even base shifts along W,
    such as the BraTS23 bundle's [0, 2, 4, 6]; or the sub-warp kernels (64-column windows with head_dim 4..32, such as the
    ISLES22 bundle's patch 4 at shifts [None, 1, 2, 3], and 8 x 16 / 128 / 256 windows) at any shifts, rank-1 HALS or MU."""
    return _core16_supported(geom, spec, relu, torch.bfloat16)


def f16_core_supported(geom: Geometry, spec: SolverSpec, relu: bool = True) -> bool:
    """The fused core takes fp16 volumes of this geometry: the same geometries as bf16_core_supported."""
    return _core16_supported(geom, spec, relu, torch.float16)


def _core16_supported(geom: Geometry, spec: SolverSpec, relu: bool, dtype: torch.dtype) -> bool:
    g, s = geom.c_geom(1, dtype), spec.c_solver()
    return bool(getattr(L.lib(), f"fz_swnmf_{_HALF[dtype]}_supported")(ctypes.byref(g), ctypes.byref(s), int(relu)))


def bf16_block_supported(x: torch.Tensor, hidden: int) -> bool:
    """FactorizerBlockBf16Fn: a contiguous, 16-byte aligned bf16 CUDA volume whose voxel count is a multiple of 8 (the bf16
    TMA boxes need 16-byte row strides), channel counts the LayerNorm kernels take (up to 512); with or without autocast.
    The caller checks the core's geometry (bf16_core_supported)."""
    return _block16_supported(x, hidden, torch.bfloat16)


def f16_block_supported(x: torch.Tensor, hidden: int) -> bool:
    """FactorizerBlockF16Fn: bf16_block_supported's conditions on an fp16 volume (fp16 autocast, or fp16 inputs).  The caller
    checks the core's geometry (f16_core_supported)."""
    return _block16_supported(x, hidden, torch.float16)


def _block16_supported(x: torch.Tensor, hidden: int, dtype: torch.dtype) -> bool:
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == dtype and x.dim() >= 3 and x.is_contiguous()
            and x.data_ptr() % 16 == 0):
        return False
    B, C = x.shape[0], x.shape[1]
    vox = x.numel() // max(B * C, 1)
    lib, H, t = L.lib(), int(hidden), _HALF[dtype]
    fwd, wgrad = getattr(lib, f"fz_linear_forward_{t}_supported"), getattr(lib, f"fz_linear_wgrad_{t}_supported")
    return bool(B > 0 and vox > 0 and getattr(lib, f"fz_layernorm_cf_{t}_supported")(C, vox)
                and fwd(C, C, vox) and fwd(H, C, vox) and fwd(C, H, vox) and wgrad(H, C, vox) and wgrad(C, H, vox))


def _staged_views(buf, shapes):
    """Per weight of shape (R, C) in `buf`, the (W, W^T) 16-bit copies fz_bf16_stage_weights / fz_f16_stage_weights wrote
    there, each as (view, row stride)."""
    views, off = [], 0
    for R, C in shapes:
        n = R * _ld8(C) + C * _ld8(R)
        views.append(((buf[off:off + R * _ld8(C)], _ld8(C)), (buf[off + R * _ld8(C):off + n], _ld8(R))))
        off += n
    return views


def _stage_weights_bf16(*ws, dtype=torch.bfloat16):
    """One launch: the fp32 matrices (one, or a block's four: the C entries take exactly those counts) as bf16 (or fp16 with
    `dtype`), each as stored and transposed; returns the buffer (see _staged_views)."""
    if len(ws) not in (1, 4):
        raise ValueError(f"factorizer_b200: 16-bit weight staging takes one or four weights, got {len(ws)}")
    lib, t = L.lib(), _HALF[dtype]
    n = sum(int(getattr(lib, f"fz_{t}_staged_elems")(w.shape[0], w.shape[1])) for w in ws)
    buf = torch.empty(n, device=ws[0].device, dtype=dtype)
    args = [a for w in ws for a in (L.ptr(w), w.shape[0], w.shape[1])]
    fn = getattr(lib, f"fz_{t}_stage_weight" if len(ws) == 1 else f"fz_{t}_stage_weights")
    _call(fn, *args, L.ptr(buf), L.stream_ptr(buf.device))
    return buf


def _channel_map_bf16(x, w, cout, bias, epi=EPI_NONE, aux=None):
    """r = W x + bias on bf16 or fp16 (B, C_in, voxels), w = (staged weight of x's dtype, row stride); returns y, or
    (y, gelu(y)) for EPI_GELU (fz_linear_forward_bf16 / _f16)."""
    B, cin, vox = x.shape
    y = torch.empty(B, cout, vox, device=x.device, dtype=x.dtype)
    y2 = torch.empty_like(y) if epi == EPI_GELU else None
    wb, ldw = w
    _call(getattr(L.lib(), f"fz_linear_forward_{_HALF[x.dtype]}"), L.ptr(x), L.ptr(wb), ldw, L.ptr(bias), L.ptr(y), B, cin, cout,
          vox, epi, L.ptr(aux), L.ptr(y2), L.stream_ptr(x.device))
    return (y, y2) if epi == EPI_GELU else y


class _Block16Fn(_WideBlockFn):
    """_WideBlockFn on 16-bit activations (`dtype` = bf16 or fp16): one launch stages the four weights in that type, as stored
    and transposed (fz_bf16_stage_weights / fz_f16_stage_weights), before the nine steps; the backward keeps the staged buffer
    and reads the transposed copies."""

    @classmethod
    def _stage(cls, ws):
        return (_stage_weights_bf16(*ws, dtype=cls.dtype),)

    @staticmethod
    def _maps(staged, shapes):
        def bind(views, shape):
            return lambda x, bias, epi=EPI_NONE, aux=None, transposed=False: _channel_map_bf16(
                x, views[transposed], shape[transposed], bias, epi, aux)
        return [bind(v, shape) for v, shape in zip(_staged_views(staged[0], shapes), shapes)]


class FactorizerBlockBf16Fn(_Block16Fn):
    """_WideBlockFn on bf16 activations: every activation (n1, z, m, x1, n2, h, g, the output, dx) is bf16 in memory and in the
    saved tensors; the parameters and their gradients stay fp32 (master weights), every sum accumulates in fp32, the
    LayerNorm statistics are fp32, and bias, residual, GELU and GELU' are applied before the one rounding to bf16.  One launch
    stages the four weights in bf16, as stored and transposed (fz_bf16_stage_weights), before the nine steps; the backward
    keeps the staged buffer and reads the transposed copies, and its weight gradients are fz_linear_wgrad_bf16."""
    dtype = torch.bfloat16

    @staticmethod
    def forward(ctx, *args):
        return FactorizerBlockBf16Fn._forward(ctx, *args)


# ---- FactorizerBlock on fp16 activations (fp16 autocast: torch.autocast("cuda")'s default, MONAI's amp) --------------
class FactorizerBlockF16Fn(_Block16Fn):
    """FactorizerBlockBf16Fn with fp16 activations: the same nine steps on the same kernels (tcgen05 kind::f16 with fp16
    operands, fz_linear_forward_f16 / fz_linear_wgrad_f16, the fp16 LayerNorm, the fp16 fused core), fp32 parameters,
    gradients and sums, one rounding to fp16 after bias, residual and GELU.  fp16 has 3 more mantissa bits than bf16 and
    a range up to 65504: a sum beyond it is stored as +-inf, which torch.amp.GradScaler detects and skips the step."""
    dtype = torch.float16

    @staticmethod
    def forward(ctx, *args):
        return FactorizerBlockF16Fn._forward(ctx, *args)


# ---- channels-first LayerNorm (glue around the mixer) --------------------------------------------
def layernorm_cf_supported(x: torch.Tensor) -> bool:
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() >= 3):
        return False
    vox = 1
    for s in x.shape[2:]:
        vox *= s
    return bool(L.lib().fz_layernorm_cf_supported(x.shape[1], vox))


class LayerNormCF(torch.autograd.Function):
    """LayerNorm over dim 1 of a (B, C, *spatial) tensor without leaving the channels-first layout
    (reference factorizer/layers/norm.py:25-34)."""

    @staticmethod
    def forward(ctx, x, weight, bias, eps: float):
        lib = L.lib()
        x = L.require_cuda_f32(x, "x")
        B, C = x.shape[0], x.shape[1]
        vox = x.numel() // max(B * C, 1)
        y = torch.empty_like(x)
        w = None if weight is None else L.require_cuda_f32(weight, "weight")
        b = None if bias is None else L.require_cuda_f32(bias, "bias")
        with torch.cuda.device(x.device):
            _call(lib.fz_layernorm_cf_forward, L.ptr(x), L.ptr(w), L.ptr(b), L.ptr(y), B, C, vox, float(eps),
                  L.stream_ptr(x.device))
        ctx.save_for_backward(x, w)
        ctx.eps, ctx.has_bias = float(eps), bias is not None
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        lib = L.lib()
        x, w = ctx.saved_tensors
        gy = L.require_cuda_f32(gy, "grad")
        B, C = x.shape[0], x.shape[1]
        vox = x.numel() // max(B * C, 1)
        gx = torch.empty_like(x)
        gw = torch.empty(C, device=x.device, dtype=torch.float32) if w is not None else None
        gb = torch.empty(C, device=x.device, dtype=torch.float32) if ctx.has_bias else None
        with torch.cuda.device(x.device):
            _call(lib.fz_layernorm_cf_backward, L.ptr(x), L.ptr(w), L.ptr(gy), L.ptr(gx), L.ptr(gw), L.ptr(gb), B, C, vox,
                  ctx.eps, L.stream_ptr(x.device))
        return gx, gw, gb, None


# ---- pointwise channel map (k = 1 Conv1d) with a hand-written weight gradient -------------------
def space_depth2_supported(x: torch.Tensor) -> bool:
    return (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and x.is_contiguous()
            and x.data_ptr() % 16 == 0 and bool(L.lib().fz_space_depth2_supported(*x.shape[2:])))


class SpaceDepth2(torch.autograd.Function):
    """to_depth: (B, C, D, H, W) -> (B, C*8, D/2*H/2*W/2), rows (c, kd, kh, kw); otherwise the inverse, taking the
    full-resolution spatial shape.  Each direction is the other's adjoint (a permutation)."""

    @staticmethod
    def forward(ctx, x, to_depth: bool, full_shape):
        B, D, H, W = x.shape[0], *full_shape
        ctx.to_depth, ctx.full_shape = to_depth, tuple(full_shape)
        return SpaceDepth2._run(x, B, D, H, W, to_depth)

    @staticmethod
    def _run(x, B, D, H, W, to_depth):
        x = L.require_cuda_f32(x, "x", allow_bf16=True)        # bf16: the scaffold's bf16 route (fz_space_depth2_bf16)
        if x.data_ptr() % 16:               # the kernel moves float4 words: the same permutation in torch
            if to_depth:
                return x.view(B, -1, D // 2, 2, H // 2, 2, W // 2, 2).permute(0, 1, 3, 5, 7, 2, 4, 6).reshape(B, -1, (D // 2) * (H // 2) * (W // 2))
            return x.view(B, -1, 2, 2, 2, D // 2, H // 2, W // 2).permute(0, 1, 5, 2, 6, 3, 7, 4).reshape(B, -1, D, H, W)
        if to_depth:
            C = x.shape[1]
            out = torch.empty(B, C * 8, (D // 2) * (H // 2) * (W // 2), device=x.device, dtype=x.dtype)
        else:
            C = x.shape[1] // 8
            out = torch.empty(B, C, D, H, W, device=x.device, dtype=x.dtype)
        fn = L.lib().fz_space_depth2_bf16 if x.dtype == torch.bfloat16 else L.lib().fz_space_depth2
        with torch.cuda.device(x.device):
            _call(fn, L.ptr(x), L.ptr(out), B, C, D, H, W, 1 if to_depth else 0, L.stream_ptr(x.device))
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        D, H, W = ctx.full_shape
        return SpaceDepth2._run(g, g.shape[0], D, H, W, not ctx.to_depth), None, None


# ---- the U-Net scaffold's layers on bf16 activations -----------------------------------------------------------------------------
def bf16_library_faster(voxels: int, out_channels: int, linear: bool) -> bool:
    """Shapes on which the library's bf16 kernels beat the bf16 route under autocast (forward + backward measured on a B200 at
    a 1000 W power limit, bench_probes/bf16_scaffold_time.py): fewer than 16 outputs (the 3-channel head at 128^3: 0.19 ms in
    cuDNN, 0.39 ms here, where a 64-output tile holds 3 outputs), and a Linear over fewer than 65536 voxels in all (the 16^3
    and 32^3 decoder adapters: 3 GEMMs against a staging launch, 3 kernels and 2 memsets; 0.79x and 0.94x).  `voxels` counts
    the whole batch."""
    return out_channels < 16 or (linear and voxels < 65536)


def bf16_layer_supported(x: torch.Tensor, voxels: int, in_channels: int, out_channels: int, linear: bool = False) -> bool:
    """The bf16 route of Linear, of the kernel-2 stride-2 and kernel-1 patch convolutions, of the transposed kernel-2 stride-2
    convolution and of the stem: a CUDA input under bf16 autocast, or a bf16 input without autocast (the FactorizerBlock
    rule); `in_channels` input channels (a mismatch falls through to the stock module, which raises); `voxels`, those of the
    channel map the layer runs per sample, a multiple of 8; a bf16 input contiguous and 16-byte aligned (an fp32 input under
    autocast is converted into a fresh buffer).  Under autocast, the shapes bf16_library_faster names keep the library
    route; a bf16 input without autocast has no other route.  fp16 autocast and fp32 without autocast keep their routes."""
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype in (torch.float32, torch.bfloat16) and x.dim() >= 3
            and x.shape[1] == in_channels):
        return False
    autocast = torch.is_autocast_enabled("cuda")
    if autocast:
        if torch.get_autocast_dtype("cuda") != torch.bfloat16:
            return False
    elif x.dtype != torch.bfloat16:
        return False
    if x.dtype == torch.bfloat16 and not (x.is_contiguous() and x.data_ptr() % 16 == 0):
        return False
    if not (x.shape[0] > 0 and 0 < int(voxels) < 2 ** 31 and int(voxels) % 8 == 0):
        return False
    return not (autocast and bf16_library_faster(x.shape[0] * int(voxels), int(out_channels), linear))


def as_bf16(x: torch.Tensor) -> torch.Tensor:
    """x as a contiguous, 16-byte aligned bf16 tensor (itself when it is one)."""
    x = x.to(torch.bfloat16, memory_format=torch.contiguous_format)
    return x if x.data_ptr() % 16 == 0 else x.clone()


class LinearBf16Fn(_GradModeFunction):
    """y = W x + b on bf16 (B, C_in, voxels) (fz_linear_forward_bf16): W = wmat, or wmat^T with `transposed` (the up-samplers'
    (C_in, C_out * K) weight read as stored).  Parameters and their gradients stay fp32, the sums are fp32 and rounded to
    bf16 once, after the bias.  One launch stages wmat in bf16 (as stored and transposed); the backward takes the other copy
    for dx and fz_linear_wgrad_bf16 for dW and db.  Saves x and the staged weight."""

    @staticmethod
    def forward(ctx, x, wmat, bias, transposed: bool):
        wmat = L.require_cuda_f32(wmat, "weight")
        bias = None if bias is None else L.require_cuda_f32(bias, "bias")
        R, C = wmat.shape
        if x.dtype != torch.bfloat16 or x.shape[1] != (R if transposed else C):
            raise ValueError(f"factorizer_b200: LinearBf16Fn takes bf16 x with {R if transposed else C} channels, got {x.dtype} "
                             f"{tuple(x.shape)}")
        with torch.cuda.device(x.device):
            staged = _stage_weights_bf16(wmat)
            w, wt = _staged_views(staged, [(R, C)])[0]
            y = _channel_map_bf16(x, wt if transposed else w, C if transposed else R, bias)
        if _GradModeFunction.wants_grad(ctx, 3):
            ctx.save_for_backward(x, staged)
            ctx.shape, ctx.transposed, ctx.has_bias = (R, C), bool(transposed), bias is not None
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        x, staged = ctx.saved_tensors
        gy = as_bf16(gy)
        w, wt = _staged_views(staged, [ctx.shape])[0]
        gx = gw = gb = None
        with torch.cuda.device(x.device):
            if ctx.needs_input_grad[0]:
                gx = _channel_map_bf16(gy, w if ctx.transposed else wt, x.shape[1], None)
            if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
                gw, gb = _channel_map_wgrad(gy, x, ctx.has_bias)
                if ctx.transposed:
                    gw = gw.t()
        return gx, gw, gb, None


def stem_bf16_supported(x: torch.Tensor, weight: torch.Tensor) -> bool:
    """StemConvBf16Fn: bf16_layer_supported, and a contiguous, 16-byte aligned x (fp32 or bf16, read as it is) of a 3x3x3
    1..4 -> 32 channel convolution with W divisible by 8 (the caller checks stride 1, padding 1, dilation, groups)."""
    if not (isinstance(x, torch.Tensor) and x.dim() == 5 and weight.dim() == 5 and tuple(weight.shape[2:]) == (3, 3, 3)
            and weight.dtype == torch.float32 and weight.is_contiguous()):
        return False
    D, H, W = x.shape[2:]
    lib = L.lib()
    return (bf16_layer_supported(x, D * H * W, weight.shape[1], weight.shape[0]) and x.is_contiguous() and x.data_ptr() % 16 == 0
            and bool(lib.fz_conv3d_stem_supported(x.shape[1], weight.shape[0], D, H, W))
            and bool(lib.fz_conv3d_stem_wgrad_bf16_supported(x.shape[1], weight.shape[0], D, H, W)))


class StemConvBf16Fn(_GradModeFunction):
    """The 3x3x3 stem with a bf16 output: x is read in the dtype it arrives in (the model's fp32 input is not converted), the
    sums are fp32 and rounded to bf16 once, after the bias (fz_conv3d_stem_forward_bf16).  The weight gradient is
    fz_conv3d_stem_wgrad_bf16, without an unfolded copy of x; dx, which the Swin Factorizer never needs, is the library's."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        B, cin, D, H, W = x.shape
        cout = weight.shape[0]
        b = None if bias is None else L.require_cuda_f32(bias.detach(), "bias")
        y = torch.empty(B, cout, D, H, W, device=x.device, dtype=torch.bfloat16)
        dt = L.FZ_DTYPE_BF16 if x.dtype == torch.bfloat16 else L.FZ_DTYPE_F32
        with torch.cuda.device(x.device):
            _call(L.lib().fz_conv3d_stem_forward_bf16, L.ptr(x), dt, L.ptr(weight.detach()), L.ptr(b), L.ptr(y), B, cin, cout, D, H, W,
                  L.stream_ptr(x.device))
        if _GradModeFunction.wants_grad(ctx):
            ctx.save_for_backward(x, weight)
            ctx.has_bias = bias is not None
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        gy = as_bf16(gy)
        B, cin, D, H, W = x.shape
        cout = weight.shape[0]
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = torch.nn.grad.conv3d_input(x.shape, weight, gy.float(), padding=1).to(x.dtype)
        if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
            gw = torch.empty_like(weight)
            gb = torch.empty(cout, device=x.device, dtype=torch.float32) if ctx.has_bias else None
            dt = L.FZ_DTYPE_BF16 if x.dtype == torch.bfloat16 else L.FZ_DTYPE_F32
            with torch.cuda.device(x.device):
                _call(L.lib().fz_conv3d_stem_wgrad_bf16, L.ptr(gy), L.ptr(x), dt, L.ptr(gw), L.ptr(gb), B, cin, cout, D, H, W,
                      L.stream_ptr(x.device))
        return gx, gw, gb


def linear_wgrad_supported(x: torch.Tensor, out_channels: int, min_voxels: int = 4096, rows: Optional[int] = None,
                           voxels: Optional[int] = None) -> bool:
    """The contraction over voxels is worth a kernel of its own when it is long (library SGEMMs take their slow
    large-K route there); short ones stay with cuBLAS."""
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() >= 3 and x.data_ptr() % 16 == 0):
        return False
    if torch.is_autocast_enabled():          # the fp32 kernels are not autocast-aware: leave mixed precision to the library
        return False
    # rows / voxels: the (B, rows, voxels) view the caller is about to build from x (space-to-depth), if not x itself
    vox = x.numel() // max(x.shape[0] * x.shape[1], 1) if voxels is None else int(voxels)
    if x.shape[0] * vox < min_voxels:
        return False
    return bool(L.lib().fz_linear_wgrad_supported(int(out_channels), x.shape[1] if rows is None else int(rows), vox))


def linear_forward(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], transposed: bool = False) -> torch.Tensor:
    """y = W x (+ b) for x (B, C_in, voxels) -- or W^T x with `transposed` (the input gradient, from the weight as stored): the
    tcgen05 channel-map kernel (csrc/fz_linear_tc.cu, 3xTF32) where its shape restrictions hold and the GEMM is large enough
    to pay, else the library's batched GEMM."""
    B, cin, vox = x.shape
    cout = weight.shape[1] if transposed else weight.shape[0]
    lib = L.lib()
    if (x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and B * vox >= 512 and cin >= 32 and cout >= 16
            and lib.fz_get_glue_mode() & 1 and lib.fz_linear_forward_supported(cout, cin, vox) and x.data_ptr() % 16 == 0
            and not (transposed and cout % 4)):
        w = weight.contiguous()
        if w.data_ptr() % 16 == 0:
            b = None if bias is None else L.require_cuda_f32(bias, "bias")
            y = torch.empty(B, cout, vox, device=x.device, dtype=torch.float32)
            with torch.cuda.device(x.device):
                _call(lib.fz_linear_forward_ex, L.ptr(x), L.ptr(w), L.ptr(b), L.ptr(y), B, cin, cout, vox, EPI_NONE, int(transposed),
                      None, None, L.stream_ptr(x.device))
            return y
    wb = (weight.t() if transposed else weight).unsqueeze(0).expand(B, -1, -1)
    return torch.bmm(wb, x) if bias is None else torch.baddbmm(bias[None, :, None], wb, x)


class LinearCF(torch.autograd.Function):
    """y = W x (+ b) over the channel axis of a (B, C_in, voxels) tensor (reference factorizer/layers/linear.py:53-58).
    Forward and input gradient: the tcgen05 channel-map kernel (linear_forward above; the library GEMM for small shapes);
    the weight / bias gradients: csrc/fz_linear_tc.cu / fz_linear.cu."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        wc = weight.contiguous()                    # a copy only for transposed views (the up-samplers' weights)
        y = linear_forward(x, wc, bias)
        ctx.save_for_backward(x, wc)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        gy = L.require_cuda_f32(gy, "grad")
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = linear_forward(gy.contiguous(), weight, None, transposed=True)
        if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
            with torch.cuda.device(x.device):                                       # gw row-major whatever the weight's strides
                gw, gb = _channel_map_wgrad(gy, x, ctx.has_bias)
        return gx, gw, gb


def stem_conv_supported(x: torch.Tensor, weight: torch.Tensor, padding) -> bool:
    """3x3x3, stride 1, padding 1, 1..4 -> 32 channels on a contiguous CUDA fp32 volume: csrc/fz_linear.cu has a direct
    kernel for the forward (the caller checks stride / dilation / groups)."""
    return (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and x.is_contiguous()
            and x.data_ptr() % 16 == 0 and weight.dim() == 5 and x.shape[1] == weight.shape[1]
            and not torch.is_autocast_enabled() and tuple(weight.shape[2:]) == (3, 3, 3) and tuple(padding) == (1, 1, 1)
            and weight.is_contiguous() and weight.dtype == torch.float32
            and bool(L.lib().fz_conv3d_stem_supported(x.shape[1], weight.shape[0], *x.shape[2:])))


def conv3d_stem_forward(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor]) -> torch.Tensor:
    B, cin, D, H, W = x.shape
    y = torch.empty(B, weight.shape[0], D, H, W, device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        _call(L.lib().fz_conv3d_stem_forward, L.ptr(x), L.ptr(weight), L.ptr(bias), L.ptr(y), B, cin, weight.shape[0], D, H, W,
              L.stream_ptr(x.device))
    return y


class ConvWgradCF(torch.autograd.Function):
    """Stride-1 convolution with few input rows (C_in * prod(kernel) <= 256: the 4 -> 32 channel 3x3x3 stem of the
    Swin Factorizer, reference factorizer/factorizer.py:139-140).  Forward and input gradient are the library's; the
    weight gradient is the channel-map kernel (csrc/fz_linear.cu) on the unfolded input, rebuilt in the backward --
    cuDNN's fp32 wgrad for that shape takes 2-4 ms at 128^3."""

    @staticmethod
    def forward(ctx, x, weight, bias, padding):
        nd = weight.dim() - 2
        if stem_conv_supported(x, weight, padding):
            y = conv3d_stem_forward(x, weight.detach(), None if bias is None else bias.detach())
        else:
            y = getattr(torch.nn.functional, f"conv{nd}d")(x, weight, bias, padding=padding)
        ctx.save_for_backward(x, weight)
        ctx.padding, ctx.has_bias = tuple(padding), bias is not None
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        import itertools
        x, weight = ctx.saved_tensors
        nd = weight.dim() - 2
        gy = L.require_cuda_f32(gy, "grad")
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = getattr(torch.nn.grad, f"conv{nd}d_input")(x.shape, weight, gy, padding=ctx.padding)
        if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
            B, cout, k, out_sp = x.shape[0], weight.shape[0], weight.shape[2:], gy.shape[2:]
            xp = torch.nn.functional.pad(x, [q for p in reversed(ctx.padding) for q in (p, p)])
            cols = torch.stack([xp[(slice(None), slice(None)) + tuple(slice(o, o + n) for o, n in zip(off, out_sp))]
                                for off in itertools.product(*[range(q) for q in k])], dim=2)   # (B, C_in, K, *out)
            with torch.cuda.device(x.device):
                gw, gb = _channel_map_wgrad(gy.view(B, cout, -1), cols.view(B, cols.shape[1] * cols.shape[2], -1), ctx.has_bias)
            gw = gw.view(weight.shape)
        return gx, gw, gb, None
