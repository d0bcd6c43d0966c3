"""ctypes binding of include/factorizer_b200.h.  There is no CPU fallback: if the shared library
is missing, or a tensor is not a CUDA float32 tensor, the call raises."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p
from typing import Optional, Sequence

import torch

from ._build import LIB_PATH

FZ_MAX_SHIFTS = 8
FZ_MAX_RANK = 8
FZ_SOLVER_MU, FZ_SOLVER_HALS = 0, 1
FZ_OK, FZ_ERR_INVALID, FZ_ERR_UNSUPPORTED, FZ_ERR_CUDA = 0, 1, 2, 3
FZ_DTYPE_F32, FZ_DTYPE_BF16, FZ_DTYPE_F16 = 0, 1, 2
FZ_PATH_AUTO, FZ_PATH_GENERIC, FZ_PATH_NO_OCTANT, FZ_PATH_OCTANT_3LAUNCH, FZ_PATH_OCTANT_PIPELINE = 0, 1, 2, 3, 4


class FzGeom(ctypes.Structure):
    _fields_ = [
        ("batch", c_int32),
        ("channels", c_int32),
        ("size", c_int32 * 3),
        ("patch", c_int32 * 3),
        ("head_dim", c_int32),
        ("num_shifts", c_int32),
        ("shifts", (c_int32 * 3) * FZ_MAX_SHIFTS),
        ("dtype", c_int32),
        ("path", c_int32),
    ]


class FzSolver(ctypes.Structure):
    _fields_ = [
        ("kind", c_int32),
        ("rank", c_int32),
        ("num_iters", c_int32),
        ("num_grad_steps", c_int32),
        ("eps", c_float),
    ]


# name -> (restype, argtypes); every symbol the header declares
_SIGNATURES = {
    "fz_version": (c_int, []),
    "fz_last_error": (c_char_p, []),
    "fz_last_path": (c_int, []),
    "fz_last_launches": (c_int, []),
    "fz_swmat_forward": (c_int, [c_void_p, c_void_p, POINTER(FzGeom), c_void_p]),
    "fz_swmat_inverse": (c_int, [c_void_p, c_void_p, POINTER(FzGeom), c_void_p]),
    "fz_swmat_forward_adjoint": (c_int, [c_void_p, c_void_p, POINTER(FzGeom), c_void_p]),
    "fz_swmat_inverse_adjoint": (c_int, [c_void_p, c_void_p, POINTER(FzGeom), c_void_p]),
    "fz_nmf_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                               c_int32, c_int32, POINTER(FzSolver), c_void_p]),
    "fz_nmf_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                c_int64, c_int32, c_int32, POINTER(FzSolver), c_void_p]),
    "fz_linear_wgrad_supported": (c_int, [c_int32, c_int32, c_int64]),
    "fz_linear_wgrad": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int64, c_void_p]),
    "fz_linear_forward_supported": (c_int, [c_int32, c_int32, c_int64]),
    "fz_linear_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int64, c_void_p]),
    "fz_linear_forward_ex": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int64, c_int32, c_int32,
                                     c_void_p, c_void_p, c_void_p]),
    "fz_conv3d_stem_supported": (c_int, [c_int32, c_int32, c_int32, c_int32, c_int32]),
    "fz_conv3d_stem_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p]),
    "fz_space_depth2_supported": (c_int, [c_int32, c_int32, c_int32]),
    "fz_space_depth2": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p]),
    "fz_space_depth2_bf16_supported": (c_int, [c_int32, c_int32, c_int32]),
    "fz_space_depth2_bf16": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p]),
    "fz_conv3d_stem_forward_bf16": (c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_int32,
                                            c_int32, c_void_p]),
    "fz_conv3d_stem_wgrad_bf16_supported": (c_int, [c_int32, c_int32, c_int32, c_int32, c_int32]),
    "fz_conv3d_stem_wgrad_bf16": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_int32,
                                          c_int32, c_void_p]),
    "fz_layernorm_cf_supported": (c_int, [c_int32, c_int64]),
    "fz_layernorm_cf_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int64, c_float, c_void_p]),
    "fz_layernorm_cf_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32,
                                         c_int64, c_float, c_void_p]),
    "fz_layernorm_cf_backward_add": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32,
                                             c_int64, c_float, c_void_p]),
    "fz_linear_forward_bf16_supported": (c_int, [c_int32, c_int32, c_int64]),
    "fz_linear_forward_bf16": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int64, c_int32,
                                       c_void_p, c_void_p, c_void_p]),
    "fz_linear_wgrad_bf16_supported": (c_int, [c_int32, c_int32, c_int64]),
    "fz_linear_wgrad_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int64, c_void_p]),
    "fz_bf16_stage_weights_supported": (c_int, [c_int32, c_int32]),
    "fz_bf16_staged_elems": (c_int64, [c_int32, c_int32]),
    "fz_bf16_stage_weights": (c_int, [c_void_p, c_int32, c_int32] * 4 + [c_void_p, c_void_p]),
    "fz_bf16_stage_weight": (c_int, [c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "fz_layernorm_cf_bf16_supported": (c_int, [c_int32, c_int64]),
    "fz_layernorm_cf_forward_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int64, c_float, c_void_p]),
    "fz_layernorm_cf_backward_add_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                                  c_int32, c_int64, c_float, c_void_p]),
    "fz_swnmf_bf16_supported": (c_int, [POINTER(FzGeom), POINTER(FzSolver), c_int32]),
    "fz_linear_forward_f16_supported": (c_int, [c_int32, c_int32, c_int64]),
    "fz_linear_forward_f16": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int64, c_int32,
                                      c_void_p, c_void_p, c_void_p]),
    "fz_linear_wgrad_f16_supported": (c_int, [c_int32, c_int32, c_int64]),
    "fz_linear_wgrad_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int64, c_void_p]),
    "fz_f16_stage_weights_supported": (c_int, [c_int32, c_int32]),
    "fz_f16_staged_elems": (c_int64, [c_int32, c_int32]),
    "fz_f16_stage_weights": (c_int, [c_void_p, c_int32, c_int32] * 4 + [c_void_p, c_void_p]),
    "fz_f16_stage_weight": (c_int, [c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "fz_layernorm_cf_f16_supported": (c_int, [c_int32, c_int64]),
    "fz_layernorm_cf_forward_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int64, c_float, c_void_p]),
    "fz_layernorm_cf_backward_add_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                                 c_int32, c_int64, c_float, c_void_p]),
    "fz_swnmf_f16_supported": (c_int, [POINTER(FzGeom), POINTER(FzSolver), c_int32]),
    "fz_set_glue_mode": (None, [c_int32]),
    "fz_get_glue_mode": (c_int, []),
    "fz_glue_supported": (c_int, [c_int32, c_int32, c_int64]),
    "fz_ln_linear_forward": (c_int, [c_void_p] * 5 + [c_int64, c_int32, c_int64, c_float, c_void_p]),
    "fz_mixer_mlp_forward": (c_int, [c_void_p] * 12 + [c_int64, c_int32, c_int32, c_int64, c_float, c_void_p]),
    "fz_mlp_backward": (c_int, [c_void_p] * 14 + [c_int64, c_int32, c_int32, c_int64, c_float, c_void_p]),
    "fz_linear_backward": (c_int, [c_void_p] * 11 + [c_int64, c_int32, c_int64, c_float, c_int32, c_void_p]),
    "fz_swnmf_saved_bytes": (c_size_t, [POINTER(FzGeom), POINTER(FzSolver)]),
    "fz_swnmf_workspace_bytes": (c_size_t, [POINTER(FzGeom), POINTER(FzSolver)]),
    "fz_swnmf_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 POINTER(FzGeom), POINTER(FzSolver), c_int32, c_void_p]),
    "fz_swnmf_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  POINTER(FzGeom), POINTER(FzSolver), c_int32, c_void_p]),
}

_lib: Optional[ctypes.CDLL] = None


def lib() -> ctypes.CDLL:
    """Load libfactorizer_b200.so (built in-tree by ``__graft_entry__.build()``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"factorizer_b200: CUDA extension not built ({LIB_PATH} missing). Run "
                "`python -c 'import __graft_entry__ as g; g.build()'` from the repo root. "
                "There is no CPU or PyTorch fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def exported_symbols() -> Sequence[str]:
    return list(_SIGNATURES)


def check(code: int) -> None:
    if code == FZ_OK:
        return
    msg = lib().fz_last_error().decode("utf-8", "replace")
    if code == FZ_ERR_UNSUPPORTED:
        raise NotImplementedError(f"factorizer_b200: {msg}")
    if code == FZ_ERR_INVALID:
        raise ValueError(f"factorizer_b200: {msg}")
    raise RuntimeError(f"factorizer_b200: {msg}")


def require_cuda_f32(t: torch.Tensor, name: str, allow_bf16: bool = False, allow_f16: bool = False) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(
            f"factorizer_b200: `{name}` is on {t.device}; this package has CUDA kernels only "
            "(no CPU fallback) - move the module and its inputs to a CUDA device")
    if t.dtype != torch.float32 and not (allow_bf16 and t.dtype == torch.bfloat16) and not (allow_f16 and t.dtype == torch.float16):
        raise NotImplementedError(
            f"factorizer_b200: `{name}` has dtype {t.dtype}; only float32 is implemented "
            "(the reference runs this path in fp32, amp: false)")
    return t.contiguous()


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def make_geom(batch: int, channels: int, size, patch, head_dim: int, shifts, path: int = 0, dtype: int = 0) -> FzGeom:
    """size/patch/shifts given for the real spatial rank (1..3); padded on the left."""
    n = len(size)
    if not 1 <= n <= 3:
        raise NotImplementedError(f"factorizer_b200: {n} spatial dims not supported (1..3)")
    if len(shifts) > FZ_MAX_SHIFTS:
        raise NotImplementedError(f"factorizer_b200: more than {FZ_MAX_SHIFTS} window sets")
    g = FzGeom()
    g.batch, g.channels, g.head_dim, g.num_shifts = batch, channels, head_dim, len(shifts)
    g.path = int(path)
    g.dtype = int(dtype)
    pad = 3 - n
    for k in range(3):
        g.size[k] = 1 if k < pad else int(size[k - pad])
        g.patch[k] = 1 if k < pad else int(patch[k - pad])
    for s, sh in enumerate(shifts):
        for k in range(3):
            g.shifts[s][k] = 0 if k < pad else int(sh[k - pad])
    return g


def make_solver(kind: int, rank: int, num_iters: int, num_grad_steps: int, eps: float) -> FzSolver:
    s = FzSolver()
    s.kind, s.rank, s.num_iters, s.num_grad_steps, s.eps = kind, rank, num_iters, num_grad_steps, eps
    return s
