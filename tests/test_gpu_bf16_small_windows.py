"""bf16 volumes on the sub-warp kernels (fz_last_path() == 3): 64-column windows with head_dim 4..32, such as the ISLES22
bundle's SWMatricize(head_dim=8, patch_size=4, shifts=[None, 1, 2, 3]) and the reference test model's num_heads=8,
patch_size=4, and 8 x 16 / 128 / 256 windows.  The window sets sum in an fp32 accumulator and y / dx are rounded to bf16
once, so the core equals the fp32 kernels' output on the same inputs, rounded by .bfloat16(), bit for bit.

1. Host-only: the support query, the refusals it keeps, and the workspace (one fp32 volume for bf16 at S >= 2; fp32 sizes
   pinned).
2. The core bit for bit against the fp32 kernels, and against the fp64 oracle at the bf16 bound (rtol 1e-2, atol 1e-3).
3. Refusals raise NotImplementedError naming the coverage.
4. FactorizerBlock at the ISLES22 geometry against the fp32 block, with the error rule of
   test_block_bf16_paired_shifts_against_fp32: only library kernels, CUDA-graph replay bit for bit.
5. Two models under bf16 autocast, with the rule of test_bundle_factorizer_under_bf16_autocast.
"""
import ctypes

import numpy as np
import pytest
import torch
from torch import nn

from conftest import assert_close
from oracle import factorizer_oracle as O
from test_gpu_fuzz import CASES as FUZZ_CASES

F = torch.nn.functional
ISLES_SHIFTS = [None, 1, 2, 3]
ISLES_RESHAPE = dict(head_dim=8, patch_size=4, shifts=ISLES_SHIFTS)

# (x shape, reshape class, reshape kwargs, solver, num_iters, num_grad_steps, relu): the ISLES22 geometry at batch 8, the
# reference test model's geometry at its widest stage, and every sub-warp case of the fuzz sweep (every M, wrap on all axes,
# MU, no ReLU, truncation, 2-D and 1-D volumes)
CORE_CASES = [
    ((8, 32, 64, 64, 64), "SWMatricize", ISLES_RESHAPE, "hals", 5, None, True),
    ((2, 256, 8, 8, 8), "SWMatricize", dict(num_heads=8, patch_size=4), "hals", 5, None, True),
] + [c[:7] for c in FUZZ_CASES if c[7] == 3]

# geometries the bf16 core still refuses: 8x512 windows whose sets do not pair up, patch 6 (generic), Matricize(grid_size=1)
# (grid-wide), rank 2
REFUSED_CASES = [
    ((1, 8, 16, 16, 16), "SWMatricize", dict(head_dim=8, patch_size=8, shifts=[None, 3, 5]), 1),
    ((1, 6, 12, 12), "SWMatricize", dict(head_dim=3, patch_size=6), 1),
    ((2, 6, 5, 9, 167), "Matricize", dict(num_heads=2, grid_size=1), 1),
    ((1, 32, 16, 16, 16), "SWMatricize", ISLES_RESHAPE, 2),
]


@pytest.fixture(scope="module")
def ft():
    from factorizer_b200 import _build
    _build.build()
    import factorizer_b200
    return factorizer_b200


def _reshape(ft, xs, cls, kw):
    return getattr(ft, cls)((None, *xs[1:]), **kw)


def _nmf(ft, reshape, solver="hals", T=5, K=None, rank=1):
    M, N = reshape.output_size[2:]
    return ft.NMF((M, N), rank=rank, num_iters=T, num_grad_steps=K, init="uniform", solver=solver)


# ---- 1. host-only -------------------------------------------------------------------------------------------------------------
def test_bf16_small_windows_support_query(ft):
    from factorizer_b200 import _ops
    for xs, cls, kw, solver, T, K, relu in CORE_CASES:
        r = _reshape(ft, xs, cls, kw)
        assert _ops.bf16_core_supported(r._geom, _nmf(ft, r, solver, T, K).solver_spec(), relu), (xs, kw)
    for C in (32, 64, 128, 256):                  # the reference test model: num_heads=8, patch 4 -> head_dim 4..32
        r = ft.SWMatricize((None, C, 16, 16, 16), num_heads=8, patch_size=4)
        assert _ops.bf16_core_supported(r._geom, _nmf(ft, r).solver_spec()), C
    for xs, cls, kw, rank in REFUSED_CASES:
        r = _reshape(ft, xs, cls, kw)
        assert not _ops.bf16_core_supported(r._geom, _nmf(ft, r, rank=rank).solver_spec()), (xs, kw, rank)


def _workspace(ft, r, spec, B, dtype):
    from factorizer_b200 import _lib
    return _lib.lib().fz_swnmf_workspace_bytes(ctypes.byref(r._geom.c_geom(B, dtype)), ctypes.byref(spec.c_solver()))


def test_bf16_small_windows_workspace(ft):
    for xs, cls, kw, solver, T, K, relu in CORE_CASES:
        r = _reshape(ft, xs, cls, kw)
        spec = _nmf(ft, r, solver, T, K).solver_spec()
        S = len(r._geom.shifts)
        b16 = _workspace(ft, r, spec, xs[0], torch.bfloat16)
        if S >= 2:
            assert b16 >= 4 * int(np.prod(xs)) and b16 % 256 == 0, (xs, kw, b16)


def test_fp32_workspace_sizes_unchanged(ft):
    """fp32 sizes as before bf16 reached the sub-warp kernels: they use no workspace; the octant and 8x512 kernels' counters"""
    sizes = []
    for xs, cls, kw, solver, T, K, relu in CORE_CASES[:2]:
        r = _reshape(ft, xs, cls, kw)
        sizes.append(_workspace(ft, r, _nmf(ft, r, solver, T, K).solver_spec(), xs[0], torch.float32))
    r = ft.SWMatricize((None, 32, 64, 64, 64), head_dim=8, patch_size=8)
    sizes.append(_workspace(ft, r, _nmf(ft, r).solver_spec(), 2, torch.float32))
    r = ft.SWMatricize((None, 8, 16, 16, 16), head_dim=8, patch_size=8, shifts=[None, 3, 5])
    sizes.append(_workspace(ft, r, _nmf(ft, r).solver_spec(), 1, torch.float32))
    assert sizes == [0, 0, 12517632, 33536], sizes


# ---- 2. the core ----------------------------------------------------------------------------------------------------------------
def _oracle(xs, cls, kw, solver, T, K, relu, nmf, x_np, gy_np):
    kwo = dict(kw)
    shifts = kwo.pop("shifts", None)
    H, d, grid, patch = O.resolve_geometry((None, *xs[1:]), **kwo)
    shifts = O.default_shifts(patch) if shifts is None else shifts
    shifts = O.normalise_shifts(shifts, len(xs) - 2)
    u0, v0 = nmf.init.u0.cpu().numpy().astype(np.float64), nmf.init.v0.cpu().numpy().astype(np.float64)
    x64, g64 = x_np.astype(np.float64), gy_np.astype(np.float64)
    y = O.swnmf_forward(x64, u0, v0, H, d, grid, patch, shifts, relu=relu, solver=solver, num_iters=T)
    gx = O.swnmf_backward(x64, g64, u0, v0, H, d, grid, patch, shifts, relu=relu, solver=solver, num_iters=T, num_grad_steps=K)
    return y, gx


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(CORE_CASES)))
def test_core_bf16_small_windows_bitwise(ft, case):
    from factorizer_b200 import _lib, _ops
    xs, cls, kw, solver, T, K, relu = CORE_CASES[case]
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(300 + case)
    r = _reshape(ft, xs, cls, kw)
    nmf = _nmf(ft, r, solver, T, K).to(dev)
    x_np = rng.standard_normal(xs).astype(np.float32)
    if solver == "mu" or not relu:                # as in test_gpu_fuzz: MU needs non-negative input
        x_np = np.abs(x_np) + np.float32(0.05)
    x = torch.from_numpy(x_np).to(dev).bfloat16()
    gy = torch.from_numpy(rng.standard_normal(xs).astype(np.float32)).to(dev).bfloat16()

    def run(v):
        v = v.clone().requires_grad_(True)
        y = _ops.SWNMF.apply(v, nmf.init.u0, nmf.init.v0, r._geom, nmf.solver_spec(), relu)
        assert _lib.lib().fz_last_path() == 3
        (gx,) = torch.autograd.grad(y, v, gy.to(v.dtype))
        assert _lib.lib().fz_last_path() == 3
        return y, gx

    y, gx = run(x)
    assert y.dtype == torch.bfloat16 and gx.dtype == torch.bfloat16
    y32, gx32 = run(x.float())
    assert torch.equal(y, y32.bfloat16()), float((y.float() - y32.bfloat16().float()).abs().max())
    assert torch.equal(gx, gx32.bfloat16()), float((gx.float() - gx32.bfloat16().float()).abs().max())
    # the oracle on the first sample (samples are independent): fp64 numpy on the whole ISLES22 batch takes minutes
    y_ref, gx_ref = _oracle((1, *xs[1:]), cls, kw, solver, T, K, relu, nmf, x[:1].float().cpu().numpy(), gy[:1].float().cpu().numpy())
    assert_close(y[:1].detach().float().cpu().numpy(), y_ref, rtol=1e-2, atol=1e-3, what="y (bf16) vs oracle")
    assert_close(gx[:1].float().cpu().numpy(), gx_ref, rtol=1e-2, atol=1e-3, what="gx (bf16) vs oracle")


# ---- 3. refusals ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(REFUSED_CASES)))
def test_core_bf16_refusals(ft, case):
    from factorizer_b200 import _ops
    xs, cls, kw, rank = REFUSED_CASES[case]
    r = _reshape(ft, xs, cls, kw)
    nmf = _nmf(ft, r, rank=rank).cuda()
    x = torch.rand(xs, device="cuda").bfloat16()
    with pytest.raises(NotImplementedError, match="sub-warp kernels"):
        _ops.SWNMF.apply(x, nmf.init.u0, nmf.init.v0, r._geom, nmf.solver_spec(), True)


# ---- 4. the block -------------------------------------------------------------------------------------------------------------------
def _block(ft, C, n, seed=3):
    torch.manual_seed(seed)
    blk = ft.FactorizerBlock(channels=C, spatial_size=(n, n, n), norm=ft.LayerNorm, reshape=(ft.SWMatricize, ISLES_RESHAPE),
                             act=nn.ReLU, factorize=ft.NMF, rank=1, num_iters=5, init="uniform", solver="hals", dropout=0.0).cuda()
    with torch.no_grad():                         # LayerNorm affine parameters away from their (1, 0) initialisation
        for ln in (blk.norm1.norm, blk.norm2.norm):
            ln.weight.add_(0.2 * torch.randn_like(ln.weight))
            ln.bias.add_(0.2 * torch.randn_like(ln.bias))
    return blk


def _run(blk, x, gout):
    blk.zero_grad(set_to_none=True)
    x = x.detach().requires_grad_(True)
    out = blk(x)
    out.backward(gout.to(out.dtype))
    return out, [x.grad] + [p.grad for p in blk.parameters()], out.grad_fn


def _parent_route(mp):
    """bf16 autocast as before the sub-warp kernels took bf16: the layers one by one, FactMixer casting the core's input"""
    from factorizer_b200 import _ops
    mp.setattr(_ops, "bf16_core_supported", lambda *a, **k: False)


def _rel(a, ref):
    return float((a.double() - ref.double()).norm() / ref.double().norm().clamp_min(1e-300))


@pytest.mark.gpu
@pytest.mark.parametrize("C,B,n", [(32, 2, 64), (64, 4, 32), (128, 8, 16), (256, 8, 8), (512, 8, 4)])
def test_block_bf16_small_windows_against_fp32(ft, monkeypatch, C, B, n):
    blk = _block(ft, C, n)
    torch.manual_seed(9)
    x = torch.randn(B, C, n, n, n, device="cuda").bfloat16()
    gout = torch.randn(B, C, n, n, n, device="cuda").bfloat16()
    out_t, grads_t, fn_t = _run(blk, x.float(), gout.float())
    assert type(fn_t).__name__ in ("FactorizerBlockFnBackward", "FactorizerBlockWideFnBackward")
    out_n, grads_n, fn_n = _run(blk, x, gout)
    assert type(fn_n).__name__ == "FactorizerBlockBf16FnBackward"
    assert out_n.dtype == torch.bfloat16 and grads_n[0].dtype == torch.bfloat16
    with monkeypatch.context() as mp:
        _parent_route(mp)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out_o, grads_o, fn_o = _run(blk, x, gout)
    assert type(fn_o).__name__ != "FactorizerBlockBf16FnBackward"
    names = ["out", "dx"] + [k for k, _ in blk.named_parameters()]
    for name, a, o, t in zip(names, [out_n] + grads_n, [out_o] + grads_o, [out_t] + grads_t):
        en, eo = _rel(a, t), _rel(o, t)
        print(f"C={C} B={B} n={n} {name}: bf16 block {en:.3g}, parent route {eo:.3g}")
        assert en <= max(1.5 * eo, 2e-3), f"{name}: relative error {en:.3g} > max(1.5 x {eo:.3g}, 2e-3)"


@pytest.mark.gpu
def test_block_bf16_small_windows_runs_only_library_kernels(ft):
    blk = _block(ft, 64, 32)
    x = torch.randn(2, 64, 32, 32, 32, device="cuda").bfloat16().requires_grad_(True)
    gout = torch.randn(2, 64, 32, 32, 32, device="cuda").bfloat16()
    blk(x).backward(gout)
    blk.zero_grad(set_to_none=True)
    x.grad = None
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = blk(x)
        out.backward(gout)
        torch.cuda.synchronize()
    assert type(out.grad_fn).__name__ == "FactorizerBlockBf16FnBackward"
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    kernels = {n for n in names if "memset" not in n.lower()}
    print(sorted(names))
    assert kernels and all("fz::" in n for n in kernels), sorted(n for n in kernels if "fz::" not in n)
    assert any("small_fwd" in n for n in kernels) and any("small_bwd" in n for n in kernels)


@pytest.mark.gpu
def test_block_bf16_small_windows_cuda_graph_replays_eager(ft):
    blk = _block(ft, 64, 32)
    x = torch.randn(4, 64, 32, 32, 32, device="cuda").bfloat16().requires_grad_(True)
    gout = torch.randn(4, 64, 32, 32, 32, device="cuda").bfloat16()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            blk.zero_grad(set_to_none=True)
            x.grad = None
            blk(x).backward(gout)
        blk.zero_grad(set_to_none=True)
        x.grad = None
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            out_g = blk(x)
            out_g.backward(gout)
    torch.cuda.current_stream().wait_stream(side)
    g.replay()
    torch.cuda.synchronize()
    got = [out_g.clone(), x.grad.clone()]
    assert type(out_g.grad_fn).__name__ == "FactorizerBlockBf16FnBackward"
    blk.zero_grad(set_to_none=True)
    x.grad = None
    out = blk(x)
    out.backward(gout)
    assert torch.equal(got[0], out) and torch.equal(got[1], x.grad)


# ---- 5. models under bf16 autocast --------------------------------------------------------------------------------------------------
def _model_under_autocast(ft, monkeypatch, net, B, n, deepest):
    """Every block takes FactorizerBlockBf16Fn but the bottleneck at `deepest`: its input reaches it from the scaffold as fp32
    under autocast, so bf16_block_supported refuses it and it runs layer by layer (the scaffold's dtype there is outside this
    change).  Errors against fp32 meet the rule of test_bundle_factorizer_under_bf16_autocast, with the parent's route (the
    bf16 core refused at patch 4) as the yardstick."""
    from factorizer_b200 import _ops
    net.train()
    torch.manual_seed(5)
    x = torch.rand(B, 4, n, n, n, device="cuda")
    target = torch.randint(0, 2, (B, 3, n, n, n), device="cuda").float()
    nodes = {}

    def hook(mod, inp, out):
        hidden = mod.mlp.block[0].linear.out_channels
        nodes[mod] = (tuple(inp[0].shape[2:]), type(out.grad_fn).__name__, _ops.bf16_block_supported(inp[0], hidden), inp[0].dtype)

    blocks = [m for m in net.modules() if isinstance(m, ft.FactorizerBlock)]
    handles = [b.register_forward_hook(hook) for b in blocks]

    def step(autocast):
        net.zero_grad(set_to_none=True)
        nodes.clear()
        torch.manual_seed(77)                     # the positional-embedding dropout draws the same masks in every run
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            logits = net(x)
        logits = logits.float()
        p = torch.sigmoid(logits)
        dice = 1 - (2 * (p * target).sum((2, 3, 4)) + 1e-5) / (p.sum((2, 3, 4)) + target.sum((2, 3, 4)) + 1e-5)
        loss = F.binary_cross_entropy_with_logits(logits, target) + dice.mean()
        loss.backward()
        return loss.detach(), [q.grad.detach().clone() if q.grad is not None else torch.zeros_like(q) for q in net.parameters()]

    truth = step(False)
    new = step(True)
    for b in blocks:
        size, fn, block_ok, dtype = nodes[b]
        print(size, fn, block_ok, dtype)
        if block_ok:
            assert fn == "FactorizerBlockBf16FnBackward", (size, fn)
        else:
            assert size == deepest and dtype == torch.float32, (size, fn, dtype)
    with monkeypatch.context() as mp:
        _parent_route(mp)
        old = step(True)
    for h in handles:
        h.remove()
    names = ["loss"] + [k for k, _ in net.named_parameters()]
    for name, a, o, t in zip(names, [new[0]] + new[1], [old[0]] + old[1], [truth[0]] + truth[1]):
        if float(t.double().norm()) == 0.0:
            continue
        en, eo = _rel(a, t), _rel(o, t)
        print(f"model {name}: bf16 blocks {en:.3g}, parent route {eo:.3g}")
        assert en <= max(1.5 * eo, 2e-3), f"{name}: relative error {en:.3g} > max(1.5 x {eo:.3g}, 2e-3)"


@pytest.mark.gpu
def test_isles22_factorizer_under_bf16_autocast(ft, monkeypatch):
    """A stand-in for the ISLES22 bundle's network: its window geometry (head_dim 8, patch 4, shifts [None, 1, 2, 3]), batch 8
    and 64^3 ROI, with the README's widths and depths (the bundle's own widths and channel counts are not recorded here)."""
    n = 64
    torch.manual_seed(1234)
    net = ft.Factorizer(in_channels=4, out_channels=3, spatial_size=(n, n, n), encoder_depth=(1, 1, 1, 1, 1),
                        encoder_width=(32, 64, 128, 256, 512), strides=(1, 2, 2, 2, 2), decoder_depth=(1, 1, 1, 1),
                        norm=ft.LayerNorm, reshape=(ft.SWMatricize, ISLES_RESHAPE), act=nn.ReLU, factorize=ft.NMF, rank=1,
                        num_iters=5, init="uniform", solver="hals", dropout=0.1).cuda()
    _model_under_autocast(ft, monkeypatch, net, 8, n, (4, 4, 4))


@pytest.mark.gpu
def test_reference_test_model_under_bf16_autocast(ft, monkeypatch):
    """The reference's tests/test_factorizer.py model: num_heads=8, patch_size=4 (head_dim 4..32), widths 32..256, 64^3."""
    n = 64
    torch.manual_seed(4321)
    net = ft.Factorizer(in_channels=4, out_channels=3, spatial_size=(n, n, n), encoder_depth=(1, 1, 1, 1),
                        encoder_width=(32, 64, 128, 256), strides=(1, 2, 2, 2), decoder_depth=(1, 1, 1),
                        norm=ft.LayerNorm, reshape=(ft.SWMatricize, dict(num_heads=8, patch_size=4)), act=nn.ReLU,
                        factorize=ft.NMF, rank=1, num_iters=5, init="uniform", solver="hals", dropout=0.1).cuda()
    _model_under_autocast(ft, monkeypatch, net, 2, n, (8, 8, 8))
