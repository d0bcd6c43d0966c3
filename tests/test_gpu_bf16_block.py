"""FactorizerBlock on bf16 activations (csrc/fz_bf16_block.cu, the bf16 LayerNorm of csrc/fz_layernorm.cu, the bf16 octant
core; _ops.FactorizerBlockBf16Fn).

1. The kernels through the C ABI against fp64 on bf16-representable inputs: the channel map (every epilogue, partial voxel
   and output tiles, 4 to 512 channels, both pipeline depths) to |y - ref| <= 2^-8 |ref| + TAU S, the weight gradient at
   production reduction lengths to TAU S, the LayerNorm forward and backward to one bf16 rounding.  S is the same sum over
   absolute values.
2. The block against the fp32 block on x.float() (itself pinned to 1e-4 by the parity tests): the relative Frobenius error
   of out, dx and every parameter gradient is at most max(1.5 x that of the layer-by-layer bf16 autocast route, 2e-3).
3. Only this library's kernels (and memsets) run; saved activations take about half the memory of the fp32 block; a CUDA
   graph replays out and dx bit for bit (the parameter gradients are atomic sums over CTAs, equal to rounding); the routes
   the bf16 path does not cover are unchanged; the Swin Factorizer under
   bf16 autocast takes the new path in every block but the 8^3 bottleneck and meets the same error rule.
"""
import math

import pytest
import torch
from torch import nn

pytestmark = pytest.mark.gpu

TAU = 2e-5
F = torch.nn.functional
EPI_NONE, EPI_RESIDUAL, EPI_GELU, EPI_GELU_GRAD, EPI_GELU_ONLY = 0, 1, 2, 3, 4


@pytest.fixture(scope="module")
def ft():
    import factorizer_b200
    return factorizer_b200


@pytest.fixture(scope="module")
def lib(ft):
    from factorizer_b200 import _lib as L
    return L.lib()


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _check(code):
    from factorizer_b200 import _lib as L
    L.check(code)


def _st():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _bf(*shape, scale=1.0, positive=False):
    t = torch.rand(*shape, device="cuda") if positive else torch.randn(*shape, device="cuda")
    return (scale * t).bfloat16()


def _gelu64(h):
    return 0.5 * h * (1.0 + torch.erf(h / math.sqrt(2.0)))


def _gelu_grad64(h):
    return 0.5 * (1.0 + torch.erf(h / math.sqrt(2.0))) + h * torch.exp(-0.5 * h * h) / math.sqrt(2.0 * math.pi)


def _ld8(n):
    return (n + 7) // 8 * 8


def _assert_bound(got, ref, S, what, rel=2.0 ** -8):
    err = (got.double() - ref).abs()
    excess = float((err - rel * ref.abs() - TAU * S).max())
    worst = float((err / (rel * ref.abs() + TAU * S).clamp_min(1e-300)).max())
    print(f"{what}: max err / (2^-8 |ref| + TAU S) = {worst:.3g}")
    assert bool(torch.isfinite(got).all()), what
    assert excess <= 0, f"{what}: max err / bound = {worst:.3g}"


# ---- 1a. channel map ---------------------------------------------------------------------------------------------------------
def _fwd_regime(sms, B, cout, cin, vox):
    items = B * -(-vox // 128) * -(-cout // 64)
    return "4-stage" if items <= sms and cin > 128 else "2-stage"


CHANNEL_MAP_CASES = {
    # name: (B, cin, cout, voxels, regime)
    "4-to-4-partial-tile": (2, 4, 4, 296, "2-stage"),
    "512-to-512": (1, 512, 512, 4096, "2-stage"),
    "256-to-60-4-stage": (1, 256, 60, 128 * 100 - 8, "4-stage"),
    "136-to-260-two-samples": (2, 136, 260, 4040, "2-stage"),
    "32-to-64-many-items": (1, 32, 64, 32 ** 3, "2-stage"),
}


@pytest.mark.parametrize("name", list(CHANNEL_MAP_CASES))
def test_channel_map_bf16_against_fp64(lib, sms, name):
    B, cin, cout, vox, regime = CHANNEL_MAP_CASES[name]
    assert _fwd_regime(sms, B, cout, cin, vox) == regime or sms != 148
    torch.manual_seed(11)
    x = _bf(B, cin, vox)
    w = _bf(cout, cin, scale=1.0 / math.sqrt(cin))
    wpad = torch.zeros(cout, _ld8(cin), device="cuda", dtype=torch.bfloat16)
    wpad[:, :cin] = w
    bias = 0.3 * torch.randn(cout, device="cuda")
    aux = _bf(B, cout, vox)
    x64, w64, a64 = x.double(), w.double(), aux.double()
    r = torch.einsum("oc,bcv->bov", w64, x64)
    S = torch.einsum("oc,bcv->bov", w64.abs(), x64.abs())
    for epi in (EPI_NONE, EPI_RESIDUAL, EPI_GELU, EPI_GELU_GRAD, EPI_GELU_ONLY):
        for b in (bias, None):
            rb = r if b is None else r + b.double()[None, :, None]
            Sb = S if b is None else S + b.double().abs()[None, :, None]
            y = torch.full((B, cout, vox), float("nan"), device="cuda", dtype=torch.bfloat16)
            y2 = torch.full_like(y, float("nan")) if epi == EPI_GELU else None
            use_aux = aux if epi in (EPI_RESIDUAL, EPI_GELU_GRAD) else None
            _check(lib.fz_linear_forward_bf16(_p(x), _p(wpad), _ld8(cin), _p(b), _p(y), B, cin, cout, vox, epi, _p(use_aux), _p(y2),
                                              _st()))
            tag = f"{name} epi={epi} bias={b is not None}"
            if epi == EPI_NONE:
                _assert_bound(y, rb, Sb, tag)
            elif epi == EPI_RESIDUAL:
                _assert_bound(y, rb + a64, Sb + a64.abs(), tag)
            elif epi == EPI_GELU:
                _assert_bound(y, rb, Sb, tag + " y")
                _assert_bound(y2, _gelu64(rb), 1.2 * Sb, tag + " gelu")
            elif epi == EPI_GELU_ONLY:
                _assert_bound(y, _gelu64(rb), 1.2 * Sb, tag)
            else:
                gp = _gelu_grad64(a64)          # gelu' is evaluated in fp32 to about 1e-6 absolute: 0.05 TAU S of slack
                _assert_bound(y, rb * gp, Sb * (gp.abs() + 0.05), tag)
    torch.cuda.synchronize()


def test_channel_map_bf16_refuses_what_it_cannot_read(lib):
    x = torch.zeros(1, 16, 64 + 8, device="cuda", dtype=torch.bfloat16)
    w = torch.zeros(16, 16, device="cuda", dtype=torch.bfloat16)
    y = torch.zeros(1, 16, 64, device="cuda", dtype=torch.bfloat16)
    from factorizer_b200 import _lib as L
    assert lib.fz_linear_forward_bf16(_p(x) + 2, _p(w), 16, None, _p(y), 1, 16, 16, 64, 0, None, None, _st()) == L.FZ_ERR_UNSUPPORTED
    assert lib.fz_linear_forward_bf16(_p(x), _p(w), 16, None, _p(y), 1, 16, 16, 60, 0, None, None, _st()) == L.FZ_ERR_UNSUPPORTED
    assert lib.fz_linear_forward_bf16(_p(x), _p(w), 12, None, _p(y), 1, 12, 16, 64, 0, None, None, _st()) == L.FZ_ERR_UNSUPPORTED
    dw = torch.zeros(16, 16, device="cuda")
    assert lib.fz_linear_wgrad_bf16(_p(x) + 2, _p(x), _p(dw), None, 1, 16, 16, 64, _st()) == L.FZ_ERR_UNSUPPORTED
    assert not lib.fz_linear_forward_bf16_supported(16, 16, 60) and lib.fz_linear_forward_bf16_supported(4, 4, 8)


# ---- 1b. weight gradient -----------------------------------------------------------------------------------------------------
WGRAD_CASES = {
    # name: (B, cout, cin, voxels)
    "64x32-over-128^3": (1, 64, 32, 128 ** 3),
    "64x64-over-2x64^3": (2, 64, 64, 64 ** 3),
    "256x128-over-32^3": (1, 256, 128, 32 ** 3),
    "512x1024-over-16^3": (1, 512, 1024, 16 ** 3),
    "60x36-partial-tiles": (3, 60, 36, 16 ** 3 + 8),
}


@pytest.mark.parametrize("data", ["zero-mean", "same-sign"])
@pytest.mark.parametrize("name", list(WGRAD_CASES))
def test_weight_gradient_bf16_against_fp64(lib, name, data):
    B, cout, cin, vox = WGRAD_CASES[name]
    torch.manual_seed(5)
    pos = data == "same-sign"
    dy, x = _bf(B, cout, vox, positive=pos), _bf(B, cin, vox, positive=pos)
    dw = torch.full((cout, cin), float("nan"), device="cuda")
    db = torch.full((cout,), float("nan"), device="cuda")
    _check(lib.fz_linear_wgrad_bf16(_p(dy), _p(x), _p(dw), _p(db), B, cout, cin, vox, _st()))
    ref = torch.zeros(cout, cin, device="cuda", dtype=torch.float64)
    S = torch.zeros_like(ref)
    for b in range(B):
        d64, x64 = dy[b].double(), x[b].double()
        ref += d64 @ x64.t()
        S += d64.abs() @ x64.abs().t()
    err = float(((dw.double() - ref).abs() / S.clamp_min(1e-300)).max())
    dbr = dy.double().sum((0, 2))
    errb = float(((db.double() - dbr).abs() / dy.double().abs().sum((0, 2)).clamp_min(1e-300)).max())
    print(f"{name} {data}: dW err/S = {err:.3g}, db err/S = {errb:.3g}")
    assert err <= TAU and errb <= TAU


# ---- 1c. LayerNorm -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,B,vox", [(32, 2, 32 ** 3), (64, 1, 64 ** 3), (64, 2, 4096), (128, 1, 32 ** 3), (256, 1, 4096),
                                     (512, 1, 4096), (100, 1, 1000)])
def test_layernorm_bf16_against_fp64(lib, C, B, vox):
    torch.manual_seed(7)
    eps = 1e-5
    x = _bf(B, C, vox, scale=2.0) + 0.5
    x = x.bfloat16()
    g, b = 1 + 0.3 * torch.randn(C, device="cuda"), 0.3 * torch.randn(C, device="cuda")
    y = torch.empty_like(x)
    _check(lib.fz_layernorm_cf_forward_bf16(_p(x), _p(g), _p(b), _p(y), B, C, vox, eps, _st()))
    xd = x.double().requires_grad_(True)
    gd, bd = g.double().requires_grad_(True), b.double().requires_grad_(True)
    yd = F.layer_norm(xd.movedim(1, -1), (C,), gd, bd, eps).movedim(-1, 1)
    xhat = F.layer_norm(x.double().movedim(1, -1), (C,), None, None, eps).movedim(-1, 1)
    scale = (g.double().abs()[None, :, None] * xhat.abs() + b.double().abs()[None, :, None])
    err = (y.double() - yd).abs()
    worst = float((err / (2.0 ** -8 * yd.abs() + 1e-5 * scale)).max())
    print(f"LN fwd C={C}: max err / (one bf16 rounding + 1e-5 scale) = {worst:.3g}")
    assert worst <= 1.0
    gy, add = _bf(B, C, vox), _bf(B, C, vox)
    dx = torch.empty_like(x)
    dg, db = torch.empty_like(g), torch.empty_like(b)
    _check(lib.fz_layernorm_cf_backward_add_bf16(_p(x), _p(g), _p(gy), _p(add), _p(dx), _p(dg), _p(db), B, C, vox, eps, _st()))
    rx, rg, rb = torch.autograd.grad((yd * gy.double()).sum(), [xd, gd, bd])
    rx = rx + add.double()
    errx = float(((dx.double() - rx).abs() / (2.0 ** -8 * rx.abs() + 1e-5 * float(rx.abs().max()))).max())
    Sg = (gy.double().abs() * xhat.abs()).sum((0, 2))
    Sb = gy.double().abs().sum((0, 2))
    errg = float(((dg.double() - rg).abs() / Sg).max())
    errb = float(((db.double() - rb).abs() / Sb).max())
    print(f"LN bwd C={C}: dx {errx:.3g}, d(gamma) err/S {errg:.3g}, d(beta) err/S {errb:.3g}")
    assert errx <= 1.0 and errg <= 1e-5 and errb <= 1e-5


# ---- 2. the block ----------------------------------------------------------------------------------------------------------------
def _block(ft, C, n, ratio, seed=3):
    torch.manual_seed(seed)
    blk = ft.FactorizerBlock(channels=C, spatial_size=(n, n, n), norm=ft.LayerNorm,
                             reshape=(ft.SWMatricize, {"head_dim": 8, "patch_size": 8}), act=nn.ReLU, factorize=ft.NMF, rank=1,
                             num_iters=5, init="uniform", solver="hals", mlp_ratio=ratio, dropout=0.0).cuda()
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


def _old_route(monkeypatch, ft):
    from factorizer_b200 import _ops
    monkeypatch.setattr(_ops, "bf16_block_supported", lambda x, hidden: False)


def _rel(a, ref):
    return float((a.double() - ref.double()).norm() / ref.double().norm().clamp_min(1e-300))


BLOCK_SHAPES = [(32, 1, 32), (64, 2, 32), (128, 1, 16), (256, 1, 16), (512, 1, 16)]


@pytest.mark.parametrize("ratio", [2, 4])
@pytest.mark.parametrize("C,B,n", BLOCK_SHAPES)
def test_block_bf16_against_fp32(ft, monkeypatch, C, B, n, ratio):
    blk = _block(ft, C, n, ratio)
    torch.manual_seed(9)
    x = torch.randn(B, C, n, n, n, device="cuda").bfloat16()
    gout = torch.randn(B, C, n, n, n, device="cuda").bfloat16()
    out_t, grads_t, fn_t = _run(blk, x.float(), gout.float())                 # fp32 truth (fused fp32 path)
    assert type(fn_t).__name__ in ("FactorizerBlockFnBackward", "FactorizerBlockWideFnBackward")
    out_n, grads_n, fn_n = _run(blk, x, gout)                                 # new bf16 path
    assert type(fn_n).__name__ == "FactorizerBlockBf16FnBackward"
    assert out_n.dtype == torch.bfloat16 and grads_n[0].dtype == torch.bfloat16
    assert all(g.dtype == torch.float32 for g in grads_n[1:])
    with monkeypatch.context() as mp:                                         # today's route under bf16 autocast
        _old_route(mp, ft)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out_o, grads_o, fn_o = _run(blk, x, gout)
    assert type(fn_o).__name__ != "FactorizerBlockBf16FnBackward"
    names = ["out", "dx"] + [k for k, _ in blk.named_parameters()]
    worst = 0.0
    for name, a, o, t in zip(names, [out_n] + grads_n, [out_o] + grads_o, [out_t] + grads_t):
        en, eo = _rel(a, t), _rel(o, t)
        bound = max(1.5 * eo, 2e-3)
        worst = max(worst, en / bound)
        print(f"C={C} n={n} ratio={ratio} {name}: new {en:.3g}, today's bf16 route {eo:.3g}, ratio {en / max(eo, 1e-300):.3g}")
        assert en <= bound, f"{name}: relative error {en:.3g} > max(1.5 x {eo:.3g}, 2e-3)"


# ---- 3. launches, memory, graphs, unchanged routes -------------------------------------------------------------------------------
def test_block_bf16_runs_only_library_kernels(ft):
    blk = _block(ft, 64, 32, 2)
    x = torch.randn(1, 64, 32, 32, 32, device="cuda").bfloat16().requires_grad_(True)
    gout = torch.randn(1, 64, 32, 32, 32, device="cuda").bfloat16()
    out = blk(x)
    out.backward(gout)
    blk.zero_grad(set_to_none=True)
    x.grad = None
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = blk(x)
        out.backward(gout)
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    kernels = {n for n in names if "memset" not in n.lower() and "Memset" not in n}
    print(sorted(names))
    assert kernels and all("fz::" in n for n in kernels), sorted(n for n in kernels if "fz::" not in n)
    assert any("linear_fwd_bf16_tc" in n for n in kernels) and any("linear_wgrad_bf16_tc" in n for n in kernels)


@pytest.mark.parametrize("C,n", [(64, 32), (128, 32), (256, 32)])
def test_block_bf16_saves_half_the_memory(ft, C, n):
    """The fixed part (the staged bf16 weights, the core's fp32 per-window records) weighs more at small volumes: 0.57 for
    256 channels at 16^3 (measured on a B200), 0.50-0.51 at 32^3 for 64, 128 and 256 channels."""
    blk = _block(ft, C, n, 2)
    x32 = torch.randn(1, C, n, n, n, device="cuda").requires_grad_(True)
    x16 = x32.detach().bfloat16().requires_grad_(True)

    def growth(x):
        blk(x).sum().backward() if x.dtype == torch.float32 else blk(x).float().sum().backward()   # workspaces exist
        blk.zero_grad(set_to_none=True)
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        out = blk(x)
        torch.cuda.synchronize()
        grow = torch.cuda.memory_allocated() - before
        del out
        return grow

    g32, g16 = growth(x32), growth(x16)
    print(f"C={C} n={n}: forward keeps {g16} bytes in bf16, {g32} in fp32: {g16 / g32:.3f}")
    assert g16 <= 0.55 * g32


def test_block_bf16_cuda_graph_replays_eager(ft):
    blk = _block(ft, 64, 32, 2)
    x = torch.randn(2, 64, 32, 32, 32, device="cuda").bfloat16().requires_grad_(True)
    gout = torch.randn(2, 64, 32, 32, 32, device="cuda").bfloat16()
    params = list(blk.parameters())
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
    got = [out_g.clone(), x.grad.clone()] + [p.grad.clone() for p in params]
    blk.zero_grad(set_to_none=True)
    x.grad = None
    out = blk(x)
    out.backward(gout)
    want = [out, x.grad] + [p.grad for p in params]
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    # the parameter gradients are sums over CTAs added with atomics, whose order is not fixed
    for a, b in zip(got[2:], want[2:]):
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-6 * float(b.abs().max()))


def test_routes_the_bf16_path_does_not_cover_are_unchanged(ft, monkeypatch):
    def both(blk, x, autocast=True):
        outs = []
        for patched in (False, True):
            with monkeypatch.context() as mp:
                if patched:
                    _old_route(mp, ft)
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                    out, grads, fn = _run(blk, x, torch.ones_like(x))
            outs.append((out, grads, type(fn).__name__))
        (a, ga, fa), (b, gb, fb) = outs
        assert fa == fb and fa != "FactorizerBlockBf16FnBackward", (fa, fb)
        assert torch.equal(a, b)
        # the layer-by-layer route's gradients include sums whose order is not fixed (atomics, library split reductions)
        for p, q in zip(ga, gb):
            assert torch.allclose(p, q, rtol=1e-5, atol=1e-6 * float(q.abs().max())), "gradient differs"

    # a geometry the bf16 core refuses: one patch along W (the 8^3 bottleneck)
    both(_block(ft, 64, 8, 2), torch.randn(1, 64, 8, 8, 8, device="cuda").bfloat16())
    # fp32 x under autocast
    blk = _block(ft, 64, 16, 2)
    both(blk, torch.randn(1, 64, 16, 16, 16, device="cuda"))
    # a bf16 x 2 bytes off a 16-byte boundary
    base = torch.randn(64 * 16 ** 3 + 1, device="cuda").bfloat16()
    xm = base[1:].view(1, 64, 16, 16, 16)
    assert xm.data_ptr() % 16 and not ft._ops.bf16_block_supported(xm, 128)
    both(blk, xm)


# ---- whole model ---------------------------------------------------------------------------------------------------------------
def test_swin_factorizer_under_bf16_autocast(ft, monkeypatch):
    n = 128
    torch.manual_seed(1234)
    net = ft.Factorizer(in_channels=4, out_channels=3, spatial_size=(n, n, n), encoder_depth=(1, 1, 1, 1, 1),
                        encoder_width=(32, 64, 128, 256, 512), strides=(1, 2, 2, 2, 2), decoder_depth=(1, 1, 1, 1),
                        norm=ft.LayerNorm, reshape=(ft.SWMatricize, {"head_dim": 8, "patch_size": 8}), act=nn.ReLU,
                        factorize=ft.NMF, rank=1, num_iters=5, init="uniform", solver="hals", mlp_ratio=2, dropout=0.1).cuda()
    net.train()
    x = torch.rand(1, 4, n, n, n, device="cuda")
    target = torch.randint(0, 2, (1, 3, n, n, n), device="cuda").float()
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
        want = "FactorizerBlockBf16FnBackward" if size != (8, 8, 8) else None
        if want:
            assert fn == want, (size, fn)
        else:
            assert fn != "FactorizerBlockBf16FnBackward", (size, fn)
    with monkeypatch.context() as mp:
        _old_route(mp, ft)
        old = step(True)
    for h in handles:
        h.remove()
    names = ["loss"] + [k for k, _ in net.named_parameters()]
    for name, a, o, t in zip(names, [new[0]] + new[1], [old[0]] + old[1], [truth[0]] + truth[1]):
        if float(t.double().norm()) == 0.0:
            continue
        en, eo = _rel(a, t), _rel(o, t)
        print(f"model {name}: new {en:.3g}, today's bf16 route {eo:.3g}")
        assert en <= max(1.5 * eo, 2e-3), f"{name}: relative error {en:.3g} > max(1.5 x {eo:.3g}, 2e-3)"
