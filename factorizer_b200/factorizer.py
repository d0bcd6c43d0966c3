"""FactMixer / FactorizerBlock / FactorizerStage: the block glue around the hot path, with the
reference's constructor signatures and parameter names (factorizer/factorizer.py:9-122).

``FactMixer.forward`` is where the fused kernel plugs in: when the configured
``reshape -> act -> factorize -> reshape.inverse_forward`` chain is
(Matricize | SWMatricize) -> (ReLU | Identity) -> NMF('mu' | 'hals'), the four steps run as the fused core (csrc/fz_swnmf_*.cu: three launches per direction on the production path);
any other combination runs the same steps through the standalone kernels.  A FactorizerBlock with LayerNorm / ReLU / GELU
and no active dropout runs entirely in hand-written kernels: 32 channels in the fused glue kernels (csrc/fz_block_glue*.cu)
around the fused core, any other width in the tcgen05 channel-map kernel with fused epilogues (csrc/fz_linear_tc.cu) and the
channels-first LayerNorm kernels, bf16 or fp16 inputs (bf16 or fp16 autocast) in the 16-bit channel maps
(csrc/fz_bf16_block.cu) around the 16-bit core (patch 8^3 at shifts [0, 4] or paired window sets such as [0, 2, 4, 6];
64-column windows such as patch 4^3 at any shifts); other blocks run the glue layer by layer.
"""
from __future__ import annotations

import torch
from torch import nn

from . import _ops
from .helpers import partialize
from .layers import MLP, LayerNorm, Linear, PositionalEmbedding
from .matrix_factorization import NMF, MatrixFactorization
from .operations import Matricize, SWMatricize

__all__ = ["FactMixer", "FactorizerBlock", "FactorizerStage"]


class FactMixer(nn.Module):
    """in_proj -> reshape -> act -> factorize -> inverse reshape -> out_proj -> dropout."""

    def __init__(self, in_channels, out_channels, spatial_size,
                 reshape=(Matricize, {"num_heads": 1, "grid_size": 1}), act=nn.ReLU, factorize=NMF,
                 dropout=0.0, **kwargs):
        super().__init__()
        self.in_proj = Linear(in_channels, out_channels, bias=False)
        self.reshape = partialize(reshape)((None, out_channels, *spatial_size))
        self.act = partialize(act)()
        self.reshaped_size = self.reshape.output_size[2:]
        self.factorize = partialize(factorize)(self.reshaped_size, **kwargs)
        # the reference passes `out_channels` as the (truthy) bias flag, factorizer.py:31
        self.out_proj = Linear(in_channels, out_channels, out_channels)
        self.dropout = nn.Dropout(dropout)

    def _fusable(self) -> bool:
        return (isinstance(self.reshape, (Matricize, SWMatricize))
                and type(self.act) in (nn.ReLU, nn.Identity)
                and isinstance(self.factorize, MatrixFactorization)
                and not self.factorize.verbose)

    def forward(self, x):
        out = self.in_proj(x)
        if self._fusable():
            f = self.factorize
            relu = isinstance(self.act, nn.ReLU)
            if out.dtype == torch.bfloat16 and not _ops.bf16_core_supported(self.reshape._geom, f.solver_spec(), relu):
                out = out.float()           # geometries the bf16 core does not cover, such as the 8^3 bottleneck at patch 8
            elif out.dtype == torch.float16 and not _ops.f16_core_supported(self.reshape._geom, f.solver_spec(), relu):
                out = out.float()           # the same for fp16
            out = _ops.SWNMF.apply(out, f.init.u0, f.init.v0, self.reshape._geom, f.solver_spec(), relu)
        else:
            out = self.reshape(out)
            out = self.act(out)
            out = self.factorize(out)
            out = self.reshape.inverse_forward(out)
        out = self.out_proj(out)
        return self.dropout(out)


class FactorizerBlock(nn.Module):
    """x + fact(norm1(x)); x + mlp(norm2(x))  (reference factorizer.py:60-77)."""

    def __init__(self, channels, spatial_size, norm=LayerNorm, dropout=0.0, mlp_ratio=2, **kwargs):
        super().__init__()
        self.norm1 = partialize(norm)(channels)
        self.fact = FactMixer(channels, channels, spatial_size, dropout=dropout, **kwargs)
        self.norm2 = partialize(norm)(channels)
        self.mlp = MLP(channels, ratio=mlp_ratio, dropout=dropout)

    def _fused_args(self, x):
        """Arguments of the fused block path, or None when this block / input is outside what it covers
        (then the layers run one by one: fused core, hand-written LayerNorm, library GEMMs)."""
        f, mlp = self.fact, self.mlp
        if not (type(self.norm1) is LayerNorm and type(self.norm2) is LayerNorm and type(mlp) is MLP
                and type(f) is FactMixer and f._fusable() and isinstance(f.act, nn.ReLU)
                and getattr(f.reshape, "_geom", None) is not None):
            return None
        n1, n2 = self.norm1.norm, self.norm2.norm
        fc1, act, dr1, fc2, dr2 = mlp.block
        drops = (f.dropout, dr1, dr2)
        if self.training and any(d.p > 0 for d in drops):
            return None
        if not (type(act) is nn.GELU and act.approximate == "none" and n1.elementwise_affine and n2.elementwise_affine
                and n1.bias is not None and n2.bias is not None and fc1.linear.bias is not None
                and fc2.linear.bias is not None and f.in_proj.linear.bias is None and f.out_proj.linear.bias is not None):
            return None
        C = x.shape[1] if x.dim() >= 3 else -1
        if tuple(n1.normalized_shape) != (C,) or tuple(n2.normalized_shape) != (C,) or fc2.linear.out_channels != C:
            return None
        if isinstance(x, torch.Tensor) and x.dtype == torch.bfloat16:
            # bf16 activations (bf16 autocast, or bf16 inputs): the bf16 channel maps around the bf16 core, where both apply
            if not (_ops.bf16_block_supported(x, fc1.linear.out_channels)
                    and _ops.bf16_core_supported(f.reshape._geom, f.factorize.solver_spec())):
                return None
            fn = _ops.FactorizerBlockBf16Fn
        elif isinstance(x, torch.Tensor) and x.dtype == torch.float16:
            # fp16 activations (fp16 autocast, or fp16 inputs): the same kernels on fp16, under the same rule
            if not (_ops.f16_block_supported(x, fc1.linear.out_channels)
                    and _ops.f16_core_supported(f.reshape._geom, f.factorize.solver_spec())):
                return None
            fn = _ops.FactorizerBlockF16Fn
        elif _ops.block_glue_supported(x, fc1.linear.out_channels):
            fn = _ops.FactorizerBlockFn            # 32 channels: fused glue kernels (csrc/fz_block_glue*.cu)
        elif _ops.wide_block_supported(x, fc1.linear.out_channels):
            fn = _ops.FactorizerBlockWideFn        # any other width: channel-map kernels with fused epilogues
        else:
            return None
        sq = lambda lin: lin.linear.weight.squeeze(-1)
        return fn, (n1.weight, n1.bias, sq(f.in_proj), sq(f.out_proj), f.out_proj.linear.bias, n2.weight, n2.bias,
                    sq(fc1), fc1.linear.bias, sq(fc2), fc2.linear.bias, f.factorize.init.u0, f.factorize.init.v0,
                    f.reshape._geom, f.factorize.solver_spec(), n1.eps, n2.eps)

    def forward(self, x):
        fused = self._fused_args(x)
        if fused is not None:
            fn, args = fused
            return fn.apply(x, *args)
        x = x + self.fact(self.norm1(x))
        x = x + self.mlp(self.norm2(x))
        return x


class FactorizerStage(nn.Module):
    """adapter -> positional embedding -> depth x FactorizerBlock (reference factorizer.py:80-122).
    As in the reference, ``dropout`` only feeds the positional-embedding dropout (:91, :101-111)."""

    def __init__(self, in_channels, out_channels, spatial_size, depth=1,
                 adapter=(Linear, {"bias": False}), pos_embed=nn.Identity, dropout=0.0, **subblocks):
        super().__init__()
        if in_channels != out_channels:
            self.adapter = partialize(adapter)(in_channels, out_channels)
        self.pos_embed = partialize(pos_embed)(out_channels, spatial_size)
        if len(list(self.pos_embed.parameters())) > 0:
            self.pos_drop = nn.Dropout(dropout)
        self.blocks = nn.ModuleList(
            FactorizerBlock(out_channels, spatial_size, **subblocks) for _ in range(depth))

    def forward(self, x):
        out = self.adapter(x) if hasattr(self, "adapter") else x
        out = self.pos_embed(out)
        if hasattr(self, "pos_drop"):
            out = self.pos_drop(out)
        for blk in self.blocks:
            out = blk(out)
        return out
