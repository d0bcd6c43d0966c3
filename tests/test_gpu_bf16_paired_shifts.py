"""bf16 volumes at window sets that pair up as (a, a + 4), such as the BraTS23 bundle's shifts [None, 2, 4, 6] (the paired
path, fz_last_path() == 4: one octant problem per pair on the volume rolled by the pair's base shift, then a roll-back-and-sum
pass in fp32 that rounds y / dx to bf16 once).

1. The core against the C oracle on the same bf16-representable inputs (rtol 1e-2 / atol 1e-3, the bound of
   test_core_bf16_activations) and against the fp32 paired kernels on the same inputs to within one bf16 rounding.
2. Refusals: an odd base shift along W, an odd number of patches along W.  The support query and the workspace size are
   host-only and run without a GPU.
3. FactorizerBlock at the bundle's shifts and mlp_ratio 4 against the fp32 block, with the error rule of
   test_block_bf16_against_fp32.
4. Only this library's kernels run, a CUDA graph replays the block bit for bit, and the bundle-configured Factorizer under
   bf16 autocast takes the bf16 block everywhere but the 8^3 bottleneck and meets the rule of
   test_swin_factorizer_under_bf16_autocast.
"""
import numpy as np
import pytest
import torch
from torch import nn

from conftest import assert_close
from oracle import c_oracle as CO

F = torch.nn.functional
BUNDLE_SHIFTS = [None, 2, 4, 6]


@pytest.fixture(scope="module")
def ft():
    from factorizer_b200 import _build
    _build.build()
    import factorizer_b200
    return factorizer_b200


def _np(t):
    return t.detach().float().cpu().numpy()


def _geom(ft, shape, shifts):
    return ft.SWMatricize((None, *shape[1:]), head_dim=8, patch_size=8, shifts=shifts)._geom


def _spec(ft, K=5):
    return ft.NMF((8, 512), rank=1, num_iters=5, num_grad_steps=K, init="uniform", solver="hals").solver_spec()


# (volume shape, shifts): both pairs at the bundle's shifts, a non-cubic volume whose second pair is rolled along every
# axis, and a geometry whose only pair is rolled
CORE_CASES = [
    ((2, 32, 64, 64, 64), BUNDLE_SHIFTS),
    ((1, 32, 128, 128, 128), BUNDLE_SHIFTS),
    ((1, 64, 16, 16, 32), [(0, 0, 0), (4, 4, 4), (2, 0, 6), (6, 4, 10)]),
    ((1, 8, 16, 16, 16), [2, 6]),
]
REFUSED_CASES = [
    ((1, 8, 16, 16, 16), [None, 1, 4, 5]),       # base shift 1 along W
    ((1, 8, 16, 16, 24), BUNDLE_SHIFTS),         # three patches along W
]


# ---- host-only ----------------------------------------------------------------------------------------------------------------
def test_bf16_paired_support_query(ft):
    from factorizer_b200 import _ops
    spec = _spec(ft)
    for shape, shifts in CORE_CASES:
        assert _ops.bf16_core_supported(_geom(ft, shape, shifts), spec), (shape, shifts)
    for shape, shifts in REFUSED_CASES:
        assert not _ops.bf16_core_supported(_geom(ft, shape, shifts), spec), (shape, shifts)


def test_bf16_paired_workspace_no_larger_than_fp32(ft):
    import ctypes

    from factorizer_b200 import _lib
    lib, s = _lib.lib(), _spec(ft).c_solver()
    for shape, shifts in CORE_CASES:
        geom = _geom(ft, shape, shifts)
        b16 = lib.fz_swnmf_workspace_bytes(ctypes.byref(geom.c_geom(shape[0], torch.bfloat16)), ctypes.byref(s))
        b32 = lib.fz_swnmf_workspace_bytes(ctypes.byref(geom.c_geom(shape[0], torch.float32)), ctypes.byref(s))
        assert 0 < b16 <= b32, (shape, shifts, b16, b32)


# ---- 1. the core -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case,K", [(0, 5), (1, 5), (2, 5), (2, 2), (3, 5)])
def test_core_bf16_paired_shifts(ft, case, K):
    from factorizer_b200 import _lib, _ops
    shape, shifts = CORE_CASES[case]
    CO.use_all_cores()
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(20 + case)
    x = torch.from_numpy(rng.standard_normal(shape, dtype=np.float32)).to(dev).bfloat16()
    gy = torch.from_numpy(rng.standard_normal(shape, dtype=np.float32)).to(dev).bfloat16()
    geom = _geom(ft, shape, shifts)
    torch.manual_seed(3)
    nmf = ft.NMF((8, 512), rank=1, num_iters=5, num_grad_steps=K, init="uniform", solver="hals").to(dev)

    def run(v):
        v = v.clone().requires_grad_(True)
        y = _ops.SWNMF.apply(v, nmf.init.u0, nmf.init.v0, geom, nmf.solver_spec(), True)
        assert _lib.lib().fz_last_path() == 4
        (gx,) = torch.autograd.grad(y, v, gy.to(v.dtype))
        assert _lib.lib().fz_last_path() == 4
        return y, gx

    y, gx = run(x)
    assert y.dtype == torch.bfloat16 and gx.dtype == torch.bfloat16
    y32, gx32 = run(x.float())
    torch.cuda.synchronize()
    v0 = _np(nmf.init.v0)
    x_np, gy_np = _np(x), _np(gy)
    y_ref = CO.swnmf_forward(x_np, v0, 8, (8, 8, 8), list(geom.shifts))
    gx_ref = CO.swnmf_backward(x_np, gy_np, v0, 8, (8, 8, 8), list(geom.shifts), num_grad_steps=K)
    assert_close(_np(y), y_ref, rtol=1e-2, atol=1e-3, what="y (bf16) vs oracle")
    assert_close(_np(gx), gx_ref, rtol=1e-2, atol=1e-3, what="gx (bf16) vs oracle")
    # the fp32 paired kernels on the same inputs: the bf16 path differs by the one rounding of the finished sum
    assert_close(_np(y), _np(y32), rtol=4e-3, atol=1e-6, what="y bf16 vs fp32 kernels")
    assert_close(_np(gx), _np(gx32), rtol=4e-3, atol=1e-3, what="gx bf16 vs fp32 kernels")


# ---- 2. refusals ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(REFUSED_CASES)))
def test_core_bf16_refuses_unpaired_geometries(ft, case):
    from factorizer_b200 import _ops
    shape, shifts = REFUSED_CASES[case]
    nmf = ft.NMF((8, 512), rank=1, num_iters=5, init="uniform", solver="hals").cuda()
    x = torch.rand(shape, device="cuda").bfloat16()
    with pytest.raises(NotImplementedError):
        _ops.SWNMF.apply(x, nmf.init.u0, nmf.init.v0, _geom(ft, shape, shifts), nmf.solver_spec(), True)


# ---- 3. the block --------------------------------------------------------------------------------------------------------------
def _block(ft, C, n, ratio=4, seed=3):
    torch.manual_seed(seed)
    blk = ft.FactorizerBlock(channels=C, spatial_size=(n, n, n), norm=ft.LayerNorm,
                             reshape=(ft.SWMatricize, {"head_dim": 8, "patch_size": 8, "shifts": BUNDLE_SHIFTS}), act=nn.ReLU,
                             factorize=ft.NMF, rank=1, num_iters=5, init="uniform", solver="hals", mlp_ratio=ratio,
                             dropout=0.0).cuda()
    with torch.no_grad():                         # LayerNorm affine parameters away from their (1, 0) initialisation
        for ln in (blk.norm1.norm, blk.norm2.norm):
            ln.weight.add_(0.2 * torch.randn_like(ln.weight))
            ln.bias.add_(0.2 * torch.randn_like(ln.bias))
    return blk


def _run(blk, x, gout):
    """out and the gradients of <out, gout>: dx, then every parameter's"""
    blk.zero_grad(set_to_none=True)
    x = x.detach().requires_grad_(True)
    out = blk(x)
    out.backward(gout.to(out.dtype))
    return out, [x.grad] + [p.grad for p in blk.parameters()], out.grad_fn


def _layer_by_layer(mp):
    """bf16 autocast without the bf16 block: the layers one by one"""
    from factorizer_b200 import _ops
    mp.setattr(_ops, "bf16_block_supported", lambda x, hidden: False)


def _rel(a, ref):
    return float((a.double() - ref.double()).norm() / ref.double().norm().clamp_min(1e-300))


@pytest.mark.gpu
@pytest.mark.parametrize("C,B,n", [(32, 2, 32), (64, 1, 32), (128, 1, 16), (256, 1, 16)])
def test_block_bf16_paired_shifts_against_fp32(ft, monkeypatch, C, B, n):
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
        _layer_by_layer(mp)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out_o, grads_o, fn_o = _run(blk, x, gout)
    assert type(fn_o).__name__ != "FactorizerBlockBf16FnBackward"
    names = ["out", "dx"] + [k for k, _ in blk.named_parameters()]
    for name, a, o, t in zip(names, [out_n] + grads_n, [out_o] + grads_o, [out_t] + grads_t):
        en, eo = _rel(a, t), _rel(o, t)
        print(f"C={C} B={B} n={n} {name}: bf16 block {en:.3g}, layer by layer {eo:.3g}")
        assert en <= max(1.5 * eo, 2e-3), f"{name}: relative error {en:.3g} > max(1.5 x {eo:.3g}, 2e-3)"


# ---- 4. kernels, graphs, model ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_block_bf16_paired_shifts_runs_only_library_kernels(ft):
    blk = _block(ft, 64, 32)
    x = torch.randn(1, 64, 32, 32, 32, device="cuda").bfloat16().requires_grad_(True)
    gout = torch.randn(1, 64, 32, 32, 32, device="cuda").bfloat16()
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
    assert any("roll_volume" in n for n in kernels) and any("unroll_combine" in n for n in kernels)


@pytest.mark.gpu
def test_block_bf16_paired_shifts_cuda_graph_replays_eager(ft):
    blk = _block(ft, 64, 32)
    x = torch.randn(2, 64, 32, 32, 32, device="cuda").bfloat16().requires_grad_(True)
    gout = torch.randn(2, 64, 32, 32, 32, device="cuda").bfloat16()
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


@pytest.mark.gpu
def test_bundle_factorizer_under_bf16_autocast(ft, monkeypatch):
    """The BraTS23 bundle's network: README widths, shifts [None, 2, 4, 6], mlp_ratio 4, batch 2, 128^3."""
    n = 128
    torch.manual_seed(1234)
    net = ft.Factorizer(in_channels=4, out_channels=3, spatial_size=(n, n, n), encoder_depth=(1, 1, 1, 1, 1),
                        encoder_width=(32, 64, 128, 256, 512), strides=(1, 2, 2, 2, 2), decoder_depth=(1, 1, 1, 1),
                        norm=ft.LayerNorm, reshape=(ft.SWMatricize, {"head_dim": 8, "patch_size": 8, "shifts": BUNDLE_SHIFTS}),
                        act=nn.ReLU, factorize=ft.NMF, rank=1, num_iters=5, init="uniform", solver="hals", mlp_ratio=4,
                        dropout=0.1).cuda()
    net.train()
    x = torch.rand(2, 4, n, n, n, device="cuda")
    target = torch.randint(0, 2, (2, 3, n, n, n), device="cuda").float()
    nodes = {}

    def hook(mod, inp, out):
        nodes[mod] = (tuple(inp[0].shape[2:]), type(out.grad_fn).__name__)

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
        size, fn = nodes[b]
        if size != (8, 8, 8):
            assert fn == "FactorizerBlockBf16FnBackward", (size, fn)
        else:
            assert fn != "FactorizerBlockBf16FnBackward", (size, fn)
    with monkeypatch.context() as mp:
        _layer_by_layer(mp)
        old = step(True)
    for h in handles:
        h.remove()
    names = ["loss"] + [k for k, _ in net.named_parameters()]
    for name, a, o, t in zip(names, [new[0]] + new[1], [old[0]] + old[1], [truth[0]] + truth[1]):
        if float(t.double().norm()) == 0.0:
            continue
        en, eo = _rel(a, t), _rel(o, t)
        print(f"model {name}: bf16 blocks {en:.3g}, layer by layer {eo:.3g}")
        assert en <= max(1.5 * eo, 2e-3), f"{name}: relative error {en:.3g} > max(1.5 x {eo:.3g}, 2e-3)"
