"""Channels-first glue layers around the hot path (SURVEY.md section 8(f) row 1).  LayerNorm runs a
hand-written channels-first kernel (csrc/fz_layernorm.cu) where it applies; Linear is a cuBLAS GEMM on the
(C_out, C_in) x (C_in, voxels) view instead of a k=1 cuDNN convolution, with its own weight-gradient kernel
(csrc/fz_linear.cu) when the contraction over voxels is long; GELU / residual adds are ATen.  Under bf16 autocast, or on bf16
inputs, Linear, the patch convolutions and the stem run this library's bf16 kernels (_ops.bf16_layer_supported).  Module and parameter names match the reference so its checkpoints load:
``Linear.linear`` (factorizer/layers/linear.py:43-58), ``LayerNorm.norm`` (layers/norm.py:25-34),
``MLP.block.{0,3}`` (layers/mlp.py:40-63), ``PositionalEmbedding.pos`` (layers/pos_embed.py:70-89).
"""
from __future__ import annotations

import math
from typing import Optional, Sequence

import torch
from torch import nn

__all__ = ["Linear", "LayerNorm", "MLP", "PositionalEmbedding", "PosEmbed", "Conv1d", "Conv2d", "Conv3d",
           "ConvTranspose1d", "ConvTranspose2d", "ConvTranspose3d"]


class Linear(nn.Module):
    """Pointwise linear map over channels of a (B, C, *spatial) tensor (a k=1 Conv1d)."""

    def __init__(self, in_channels: int, out_channels: int, bias: bool = True, device=None, dtype=None):
        super().__init__()
        self.flatten = nn.Flatten(start_dim=2)
        self.linear = nn.Conv1d(in_channels, out_channels, kernel_size=1, bias=bias, device=device,
                                dtype=dtype)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        # same arithmetic as the k=1 Conv1d of the reference (layers/linear.py:53-58), as one GEMM per
        # sample: W (C_out, C_in) @ x (C_in, voxels); the Conv1d module only holds the parameters
        shape = x.shape
        w = self.linear.weight.squeeze(-1)
        xf = self.flatten(x)                                  # (B, C_in, voxels): a view, no copy
        from . import _ops
        if _ops.bf16_layer_supported(x, xf.shape[-1], w.shape[1], w.shape[0], linear=True):
            # bf16 autocast, or bf16 x: bf16 tensor-core channel map (csrc/fz_bf16_block.cu), fp32 parameters
            return _ops.LinearBf16Fn.apply(_ops.as_bf16(xf), w, self.linear.bias, False).view(shape[0], -1, *shape[2:])
        if torch.is_grad_enabled() and w.requires_grad and xf.is_contiguous() and _ops.linear_wgrad_supported(xf, w.shape[0]):
            # long contractions over voxels: hand-written weight-gradient kernel (csrc/fz_linear.cu)
            return _ops.LinearCF.apply(xf, w, self.linear.bias).view(shape[0], -1, *shape[2:])
        if xf.is_cuda and xf.dtype == torch.float32 and not torch.is_autocast_enabled() and not (torch.is_grad_enabled() and (w.requires_grad or xf.requires_grad)):
            # inference: the same kernel choice as the differentiable path (tcgen05 channel map where it applies)
            y = _ops.linear_forward(xf.contiguous(), w, self.linear.bias)
        elif self.linear.bias is not None:
            y = torch.baddbmm(self.linear.bias[None, :, None], w.unsqueeze(0).expand(shape[0], -1, -1), xf)
        else:
            y = torch.bmm(w.unsqueeze(0).expand(shape[0], -1, -1), xf)
        return y.view(shape[0], -1, *shape[2:])


class _PatchConv:
    """Mixin for nn.ConvNd: a convolution over non-overlapping patches (kernel_size == stride, no padding -- the
    reference U-Net's strided down-samplers, factorizer/unet.py:53, and its 1x1 head, unet.py:247) is a pointwise
    channel map on the space-to-depth view of the input.  On CUDA fp32 tensors it runs as one (a library GEMM
    forward, 0.3 ms instead of cuDNN's 0.54 ms for the first down-sampler), so that its weight gradient comes from
    csrc/fz_linear.cu instead of cuDNN's fp32 wgrad (1.7 ms per layer at 128^3); every other convolution shape is the
    stock nn.ConvNd.  Parameters and state_dict
    keys are those of nn.ConvNd."""

    def _patch_view(self, x: torch.Tensor):
        k = self.kernel_size
        if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == len(k) + 2 and self.groups == 1
                and tuple(self.stride) == tuple(k) and all(d == 1 for d in self.dilation)
                and not isinstance(self.padding, str) and all(p == 0 for p in self.padding)
                and all(n % q == 0 for n, q in zip(x.shape[2:], k))):
            return None
        B, C = x.shape[:2]
        out_sp = [n // q for n, q in zip(x.shape[2:], k)]
        from . import _ops
        if not _ops.linear_wgrad_supported(x, self.out_channels, min_voxels=64, rows=C * math.prod(k), voxels=math.prod(out_sp)):
            return None
        if all(q == 1 for q in k):
            xf = x.reshape(B, C, -1)
        elif tuple(k) == (2, 2, 2) and _ops.space_depth2_supported(x):
            xf = _ops.SpaceDepth2.apply(x, True, tuple(x.shape[2:]))                         # hand-written permutation
        else:
            split = [d for n, q in zip(out_sp, k) for d in (n, q)]
            nd = len(k)
            perm = [0, 1] + [3 + 2 * i for i in range(nd)] + [2 + 2 * i for i in range(nd)]
            xf = x.reshape(B, C, *split).permute(perm).reshape(B, C * math.prod(k), -1)     # (ci, k...) rows, one copy
        if not xf.is_contiguous():
            xf = xf.contiguous()
        return xf, out_sp

    def _unfold_ok(self, x: torch.Tensor) -> bool:
        """Stride-1 convolution whose unfolded input has few rows (the 4 -> 32 channel stem): library forward,
        weight gradient from csrc/fz_linear.cu on the unfolded input (see _ops.ConvWgradCF)."""
        k = self.kernel_size
        if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == len(k) + 2 and torch.is_grad_enabled()
                and self.weight.requires_grad and self.groups == 1 and all(q == 1 for q in self.stride)
                and all(d == 1 for d in self.dilation) and not isinstance(self.padding, str)
                and self.padding_mode == "zeros" and math.prod(k) > 1 and x.is_contiguous()
                and not torch.is_autocast_enabled()):
            return False
        rows = self.in_channels * math.prod(k)
        out_sp = [n + 2 * p - q + 1 for n, p, q in zip(x.shape[2:], self.padding, k)]
        vox = math.prod(out_sp)
        # the unfolded copy is rows * voxels floats: keep it under 2 GiB
        return (rows <= 256 and min(out_sp) > 0 and vox % 4 == 0 and x.shape[0] * vox >= 4096
                and x.shape[0] * rows * vox * 4 <= 2 ** 31)

    def _bf16_forward(self, x: torch.Tensor):
        """The bf16 route (_ops.bf16_layer_supported): the 3-D kernel-2 stride-2 down-sampler as bf16 space-to-depth + the bf16
        channel map, a kernel-1 convolution as the bf16 channel map on the flattened view, the 3x3x3 stem as StemConvBf16Fn;
        None for every other layer or shape."""
        from . import _ops
        k, sp = tuple(self.kernel_size), tuple(x.shape[2:])
        if not (x.dim() == len(k) + 2 and self.groups == 1 and all(d == 1 for d in self.dilation) and not isinstance(self.padding, str)
                and self.padding_mode == "zeros"):
            return None
        B, C, co = x.shape[0], x.shape[1], self.out_channels
        if tuple(self.stride) == k and all(p == 0 for p in self.padding):
            out_sp = [n // q for n, q in zip(sp, k)]
            if all(q == 1 for q in k):
                if not _ops.bf16_layer_supported(x, math.prod(sp), self.in_channels, co):
                    return None
                xf = _ops.as_bf16(x).view(B, C, -1)
            elif k == (2, 2, 2) and _ops.L.lib().fz_space_depth2_bf16_supported(*sp) and _ops.bf16_layer_supported(x, math.prod(out_sp), self.in_channels, co):
                xf = _ops.SpaceDepth2.apply(_ops.as_bf16(x), True, sp)                             # bf16 permutation
            else:
                return None
            y = _ops.LinearBf16Fn.apply(xf, self.weight.reshape(co, -1), self.bias, False)
            return y.view(B, co, *out_sp)
        if (k == (3, 3, 3) and all(q == 1 for q in self.stride) and tuple(self.padding) == (1, 1, 1)
                and _ops.stem_bf16_supported(x, self.weight)):
            return _ops.StemConvBf16Fn.apply(x, self.weight, self.bias)
        return None

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        pv = self._patch_view(x)
        if pv is None:
            from . import _ops
            y = self._bf16_forward(x)
            if y is not None:
                return y
            if self._unfold_ok(x):
                return _ops.ConvWgradCF.apply(x, self.weight, self.bias, tuple(self.padding))
            if (not (torch.is_grad_enabled() and (x.requires_grad or self.weight.requires_grad)) and self.groups == 1
                    and all(q == 1 for q in self.stride) and all(q == 1 for q in self.dilation)
                    and not isinstance(self.padding, str) and self.padding_mode == "zeros"
                    and _ops.stem_conv_supported(x, self.weight, self.padding)):
                return _ops.conv3d_stem_forward(x, self.weight, self.bias)       # inference: direct stem kernel
            return super().forward(x)
        from . import _ops
        xf, out_sp = pv
        y = _ops.LinearCF.apply(xf, self.weight.reshape(self.out_channels, -1), self.bias)
        return y.view(x.shape[0], self.out_channels, *out_sp)


class Conv1d(_PatchConv, nn.Conv1d):
    pass


class Conv2d(_PatchConv, nn.Conv2d):
    pass


class Conv3d(_PatchConv, nn.Conv3d):
    pass


class _PatchConvTranspose:
    """Mixin for nn.ConvTransposeNd: with kernel_size == stride and no padding (the reference U-Net's up-samplers,
    factorizer/unet.py:97-99) every input voxel writes its own output patch, i.e. the layer is a pointwise channel map
    C_in -> C_out * prod(kernel) followed by a depth-to-space permutation.  Same conditions and purpose as _PatchConv."""

    def _patch_ok(self, x: torch.Tensor) -> bool:
        k = self.kernel_size
        if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == len(k) + 2 and self.groups == 1
                and tuple(self.stride) == tuple(k) and all(d == 1 for d in self.dilation)
                and all(p == 0 for p in self.padding) and all(p == 0 for p in self.output_padding) and x.is_contiguous()):
            return False
        from . import _ops
        return _ops.linear_wgrad_supported(x.flatten(2), self.out_channels * math.prod(k), min_voxels=64)

    def _bf16_forward(self, x: torch.Tensor):
        """The bf16 route (_ops.bf16_layer_supported) of the 3-D kernel-2 stride-2 up-sampler: the bf16 channel map with the
        transposed staged weight (rows (co, k)), then bf16 depth-to-space; None for every other layer or shape."""
        from . import _ops
        k = tuple(self.kernel_size)
        if not (k == (2, 2, 2) and x.dim() == 5 and self.groups == 1 and tuple(self.stride) == k and all(d == 1 for d in self.dilation)
                and all(p == 0 for p in self.padding) and all(p == 0 for p in self.output_padding)):
            return None
        full = tuple(2 * n for n in x.shape[2:])
        if not (_ops.L.lib().fz_space_depth2_bf16_supported(*full) and _ops.bf16_layer_supported(x, math.prod(x.shape[2:]), self.in_channels, self.out_channels * 8)):
            return None
        B, co, K = x.shape[0], self.out_channels, math.prod(k)
        w = self.weight.reshape(self.in_channels, co * K)                        # (ci, (co, k)) as stored
        b = None if self.bias is None else self.bias.repeat_interleave(K)
        y = _ops.LinearBf16Fn.apply(_ops.as_bf16(x).view(B, x.shape[1], -1), w, b, True)
        return _ops.SpaceDepth2.apply(y, False, full)                           # bf16 permutation

    def forward(self, x: torch.Tensor, output_size=None) -> torch.Tensor:
        if output_size is None:
            y = self._bf16_forward(x)
            if y is not None:
                return y
        if output_size is not None or not self._patch_ok(x):
            return super().forward(x, output_size)
        from . import _ops
        k, nd = self.kernel_size, len(self.kernel_size)
        B, co, K = x.shape[0], self.out_channels, math.prod(self.kernel_size)
        w = self.weight.reshape(self.in_channels, co * K).t()                   # rows (co, k...), a view
        b = None if self.bias is None else self.bias.repeat_interleave(K)
        y = _ops.LinearCF.apply(x.flatten(2), w, b)                             # (B, co * K, voxels)
        sp = x.shape[2:]
        full = [n * q for n, q in zip(sp, k)]
        if tuple(k) == (2, 2, 2) and full[2] % 4 == 0:
            return _ops.SpaceDepth2.apply(y, False, tuple(full))                # hand-written permutation
        perm = [0, 1] + [d for i in range(nd) for d in (2 + nd + i, 2 + i)]
        y = y.view(B, co, *k, *sp).permute(perm)                                # (B, co, n0, k0, n1, k1, ...)
        return y.reshape(B, co, *[n * q for n, q in zip(sp, k)])                # one copy


class ConvTranspose1d(_PatchConvTranspose, nn.ConvTranspose1d):
    pass


class ConvTranspose2d(_PatchConvTranspose, nn.ConvTranspose2d):
    pass


class ConvTranspose3d(_PatchConvTranspose, nn.ConvTranspose3d):
    pass


class LayerNorm(nn.Module):
    """LayerNorm over the channel axis of a channels-first tensor."""

    def __init__(self, dim: int, **kwargs):
        super().__init__()
        self.norm = nn.LayerNorm(dim, **kwargs)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        from . import _ops
        if _ops.layernorm_cf_supported(x) and tuple(self.norm.normalized_shape) == (x.shape[1],):
            return _ops.LayerNormCF.apply(x, self.norm.weight, self.norm.bias, self.norm.eps)
        y = self.norm(x.movedim(1, -1))
        return y.movedim(-1, 1)


class MLP(nn.Module):
    """Linear -> GELU -> Dropout -> Linear -> Dropout (reference default ratio 3.0, mlp.py:45)."""

    def __init__(self, in_channels: int, out_channels: Optional[int] = None,
                 hidden_channels: Optional[int] = None, ratio: float = 3.0, dropout=0.0, **kwargs):
        super().__init__()
        out_channels = out_channels or in_channels
        hidden_channels = hidden_channels or int(ratio * in_channels)
        p = tuple(dropout) if isinstance(dropout, (tuple, list)) else (dropout, dropout)
        self.block = nn.Sequential(
            Linear(in_channels, hidden_channels, **kwargs),
            nn.GELU(),
            nn.Dropout(p[0]),
            Linear(hidden_channels, out_channels, **kwargs),
            nn.Dropout(p[1]),
        )

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self.block(x)


class PositionalEmbedding(nn.Module):
    """Learnable additive positional embedding (1, C, *spatial)."""

    def __init__(self, channels: int, spatial_size: Sequence[int]) -> None:
        super().__init__()
        self.pos = nn.Parameter(torch.empty(1, channels, *spatial_size))
        nn.init.normal_(self.pos, std=1.0)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return x + self.pos


PosEmbed = PositionalEmbedding
