"""The U-Net scaffold's layers on bf16 activations (_ops.bf16_layer_supported, LinearBf16Fn, StemConvBf16Fn, the bf16
space-to-depth and stem kernels of csrc/fz_linear.cu, the stem weight gradient of csrc/fz_bf16_block.cu).

1. The kernels through the C ABI: the bf16 space-to-depth bit for bit against the torch permutation; the stem forward and its
   weight gradient against fp64 on bf16-representable inputs, with the bounds of test_gpu_bf16_block.py (outputs within
   2^-8 |ref| + TAU S, weight and bias gradients within TAU S, S the same contraction over absolute values).
2. Each layer under bf16 autocast (fp32 input) and on bf16 input without autocast: bf16 output, fp32 parameter gradients, the
   new autograd node, and the same fp64 bounds.
3. The Swin Factorizer at 128^3 under bf16 autocast against the fp32 run, with the library-route scaffold as the yardstick;
   which kernels run; CUDA-graph replay; the routes this does not cover are unchanged.
"""
import copy
import math

import pytest
import torch
from torch import nn

pytestmark = pytest.mark.gpu

TAU = 2e-5
F = torch.nn.functional


@pytest.fixture(scope="module")
def ft():
    import factorizer_b200
    return factorizer_b200


@pytest.fixture(scope="module")
def lib(ft):
    from factorizer_b200 import _lib as L
    return L.lib()


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


def _assert_bound(got, ref, S, what, rel=2.0 ** -8):
    err = (got.double() - ref).abs()
    worst = float((err / (rel * ref.abs() + TAU * S).clamp_min(1e-300)).max())
    print(f"{what}: max err / (2^-8 |ref| + TAU S) = {worst:.3g}")
    assert bool(torch.isfinite(got).all()), what
    assert worst <= 1.0, f"{what}: max err / bound = {worst:.3g}"


# ---- 1. kernels ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,C,D,H,W", [(1, 32, 128, 128, 128), (3, 8, 64, 32, 48)])
def test_space_depth2_bf16_is_the_permutation(lib, B, C, D, H, W):
    torch.manual_seed(1)
    x = _bf(B, C, D, H, W)
    rows = torch.empty(B, C * 8, (D // 2) * (H // 2) * (W // 2), device="cuda", dtype=torch.bfloat16)
    _check(lib.fz_space_depth2_bf16(_p(x), _p(rows), B, C, D, H, W, 1, _st()))
    ref = x.view(B, C, D // 2, 2, H // 2, 2, W // 2, 2).permute(0, 1, 3, 5, 7, 2, 4, 6).reshape(rows.shape)
    assert torch.equal(rows, ref)
    # the other direction on independent data, and the adjoint identity <S x, y> = <x, S^T y>
    y = _bf(*rows.shape)
    back = torch.empty_like(x)
    _check(lib.fz_space_depth2_bf16(_p(y), _p(back), B, C, D, H, W, 0, _st()))
    assert torch.equal(back, y.view(B, C, 2, 2, 2, D // 2, H // 2, W // 2).permute(0, 1, 5, 2, 6, 3, 7, 4).reshape(x.shape))
    assert math.isclose(float((rows.double() * y.double()).sum()), float((x.double() * back.double()).sum()), rel_tol=1e-12)


@pytest.mark.parametrize("xdt", ["fp32", "bf16"])
@pytest.mark.parametrize("cin", [1, 2, 3, 4])
def test_stem_forward_bf16_against_fp64(lib, cin, xdt):
    from factorizer_b200 import _lib as L
    torch.manual_seed(2 + cin)
    B, D, H, W = 2, 12, 20, 32
    x = _bf(B, cin, D, H, W)
    w = torch.randn(32, cin, 3, 3, 3, device="cuda") / math.sqrt(27 * cin)
    b = 0.3 * torch.randn(32, device="cuda")
    xin, dt = (x.float(), L.FZ_DTYPE_F32) if xdt == "fp32" else (x, L.FZ_DTYPE_BF16)
    for bias in (b, None):
        y = torch.full((B, 32, D, H, W), float("nan"), device="cuda", dtype=torch.bfloat16)
        _check(lib.fz_conv3d_stem_forward_bf16(_p(xin), dt, _p(w), _p(bias), _p(y), B, cin, 32, D, H, W, _st()))
        b64 = None if bias is None else bias.double()
        ref = F.conv3d(x.double(), w.double(), b64, padding=1)
        S = F.conv3d(x.double().abs(), w.double().abs(), None if bias is None else b64.abs(), padding=1)
        _assert_bound(y, ref, S, f"stem cin={cin} x={xdt} bias={bias is not None}")


STEM_WGRAD_CASES = {
    # name: (B, cin, D, H, W, x dtype)
    "4ch-128^3-fp32-x": (1, 4, 128, 128, 128, "fp32"),
    "3ch-odd-batch-bf16-x": (3, 3, 10, 12, 24, "bf16"),
    "1ch-fp32-x": (2, 1, 16, 8, 40, "fp32"),
    "2ch-partial-tile-bf16-x": (3, 2, 3, 5, 8, "bf16"),        # 120 voxels: the last 64-voxel tile is partly past the volume
}


@pytest.mark.parametrize("data", ["zero-mean", "same-sign"])
@pytest.mark.parametrize("name", list(STEM_WGRAD_CASES))
def test_stem_weight_gradient_bf16_against_fp64(lib, name, data):
    from factorizer_b200 import _lib as L
    B, cin, D, H, W, xdt = STEM_WGRAD_CASES[name]
    torch.manual_seed(4)
    pos = data == "same-sign"
    x, dy = _bf(B, cin, D, H, W, positive=pos), _bf(B, 32, D, H, W, positive=pos)
    xin, dt = (x.float(), L.FZ_DTYPE_F32) if xdt == "fp32" else (x, L.FZ_DTYPE_BF16)
    dw = torch.full((32, cin, 3, 3, 3), float("nan"), device="cuda")
    db = torch.full((32,), float("nan"), device="cuda")
    _check(lib.fz_conv3d_stem_wgrad_bf16(_p(dy), _p(xin), dt, _p(dw), _p(db), B, cin, 32, D, H, W, _st()))
    x64, d64 = x.double(), dy.double()
    ref = torch.nn.grad.conv3d_weight(x64, dw.shape, d64, padding=1)
    S = torch.nn.grad.conv3d_weight(x64.abs(), dw.shape, d64.abs(), padding=1)
    err = float(((dw.double() - ref).abs() / S.clamp_min(1e-300)).max())
    errb = float(((db.double() - d64.sum((0, 2, 3, 4))).abs() / d64.abs().sum((0, 2, 3, 4))).max())
    print(f"{name} {data}: dW err/S = {err:.3g}, db err/S = {errb:.3g}")
    assert err <= TAU and errb <= TAU


def test_bf16_scaffold_kernels_refuse_what_they_cannot_read(lib):
    from factorizer_b200 import _lib as L
    x = torch.zeros(4 * 8 * 8 * 16 + 8, device="cuda", dtype=torch.bfloat16)
    out = torch.zeros_like(x)
    w = torch.zeros(32, 4, 3, 3, 3, device="cuda")
    dw = torch.zeros_like(w)
    U = L.FZ_ERR_UNSUPPORTED
    assert lib.fz_space_depth2_bf16(_p(x) + 2, _p(out), 1, 4, 8, 8, 16, 1, _st()) == U
    assert lib.fz_space_depth2_bf16(_p(x), _p(out) + 8, 1, 4, 8, 8, 16, 0, _st()) == U
    assert lib.fz_space_depth2_bf16(_p(x), _p(out), 1, 4, 8, 8, 6, 1, _st()) == U
    assert lib.fz_conv3d_stem_forward_bf16(_p(x) + 2, L.FZ_DTYPE_BF16, _p(w), None, _p(out), 1, 4, 32, 8, 8, 16, _st()) == U
    assert lib.fz_conv3d_stem_wgrad_bf16(_p(x) + 2, _p(x), L.FZ_DTYPE_BF16, _p(dw), None, 1, 4, 32, 8, 8, 16, _st()) == U
    assert lib.fz_conv3d_stem_wgrad_bf16(_p(x), _p(x) + 4, L.FZ_DTYPE_BF16, _p(dw), None, 1, 4, 32, 8, 8, 16, _st()) == U
    assert lib.fz_conv3d_stem_wgrad_bf16(_p(x), _p(x), L.FZ_DTYPE_BF16, _p(dw), None, 1, 4, 32, 8, 8, 12, _st()) == U
    assert not lib.fz_conv3d_stem_wgrad_bf16_supported(4, 32, 8, 8, 12) and lib.fz_conv3d_stem_wgrad_bf16_supported(4, 32, 8, 8, 16)
    assert not lib.fz_space_depth2_bf16_supported(8, 8, 6) and lib.fz_space_depth2_bf16_supported(8, 8, 4)
    torch.cuda.synchronize()


# ---- 2. layers -------------------------------------------------------------------------------------------------------------------
def _layer(ft, name):
    from factorizer_b200 import layers
    torch.manual_seed(6)
    mod, shape = {
        "linear": (lambda: ft.Linear(48, 40), (2, 48, 32, 32, 32)),
        "down-k2s2": (lambda: layers.Conv3d(32, 64, kernel_size=2, stride=2), (2, 32, 16, 16, 32)),
        "up-k2s2": (lambda: layers.ConvTranspose3d(64, 32, kernel_size=2, stride=2), (2, 64, 8, 8, 8)),
        "head-k1": (lambda: layers.Conv3d(32, 3, kernel_size=1), (2, 32, 16, 16, 16)),
        "stem": (lambda: layers.Conv3d(4, 32, kernel_size=3, padding=1), (2, 4, 5, 6, 16)),      # 480 voxels: a partial tile
    }[name]
    m = mod().cuda()
    with torch.no_grad():                                 # bf16-representable parameters: the fp64 reference is exact
        for p in m.parameters():
            p.copy_(p.bfloat16().float())
    return m, shape


ROUTE = ("LinearBf16FnBackward", "StemConvBf16FnBackward")


def _node_names(t, depth=3):
    names, frontier = set(), [t.grad_fn]
    for _ in range(depth):
        nxt = []
        for fn in frontier:
            if fn is not None:
                names.add(type(fn).__name__)
                nxt += [f for f, _ in fn.next_functions]
        frontier = nxt
    return names


LAYERS = ["linear", "down-k2s2", "up-k2s2", "head-k1", "stem"]


@pytest.mark.parametrize("mode", ["autocast", "bf16-input"])
@pytest.mark.parametrize("name", LAYERS)
def test_layer_bf16_against_fp64(ft, monkeypatch, name, mode):
    from factorizer_b200 import _ops
    m, shape = _layer(ft, name)
    x16 = _bf(*shape)
    x = (x16.float() if mode == "autocast" else x16).requires_grad_(True)
    # the kernels on every layer, including the head the speed rule leaves to the library under autocast
    monkeypatch.setattr(_ops, "bf16_library_faster", lambda *a, **k: False)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=mode == "autocast"):
        y = m(x)
    assert y.dtype == torch.bfloat16
    want = "StemConvBf16FnBackward" if name == "stem" else "LinearBf16FnBackward"
    assert want in _node_names(y), _node_names(y)
    gy = _bf(*y.shape)
    y.backward(gy)
    assert all(p.grad.dtype == torch.float32 for p in m.parameters())
    # fp64 truth, and S from the same layer with |parameters| on |x|, |gy|
    m64, a64 = copy.deepcopy(m).double(), copy.deepcopy(m).double()
    with torch.no_grad():
        for p in a64.parameters():
            p.abs_()
    xr = x16.detach().double().requires_grad_(True)
    ref = m64(xr)
    ref.backward(gy.double())
    xa = x16.detach().double().abs().requires_grad_(True)
    S = a64(xa)
    S.backward(gy.double().abs())
    _assert_bound(y, ref.detach(), S.detach(), f"{name} {mode} out")
    _assert_bound(x.grad, xr.grad, xa.grad, f"{name} {mode} dx")
    for (k, p), p64, pa in zip(m.named_parameters(), m64.parameters(), a64.parameters()):
        err = float(((p.grad.double() - p64.grad).abs() / pa.grad.clamp_min(1e-300)).max())
        print(f"{name} {mode} d{k}: err/S = {err:.3g}")
        assert err <= TAU, k


# ---- 3. routes that do not change ------------------------------------------------------------------------------------------------
def test_autocast_keeps_the_library_where_it_is_faster(ft):
    """Under bf16 autocast the head (3 outputs) and a Linear over fewer than 65536 voxels keep the stock route
    (_ops.bf16_library_faster); on bf16 input without autocast, where the stock modules raise, they take the bf16 route."""
    m, shape = _layer(ft, "head-k1")
    small = ft.Linear(48, 40).cuda()
    for mod, x in ((m, torch.randn(*shape, device="cuda")), (small, torch.randn(2, 48, 8, 8, 16, device="cuda"))):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = mod(x)
            assert not any(k in ROUTE for k in _node_names(y)) and torch.equal(y, _stock(mod, x)), type(mod).__name__
        y = mod(x.bfloat16())
        assert y.dtype == torch.bfloat16 and "LinearBf16FnBackward" in _node_names(y), type(mod).__name__


def test_channel_mismatch_falls_through_to_the_stock_module(ft):
    """A wrong channel count takes no kernel of this library (which would read the weight with the wrong shape): the stock
    module raises, as it does on every other route."""
    for name, cin in (("linear", 32), ("down-k2s2", 16), ("up-k2s2", 48), ("head-k1", 16), ("stem", 3)):
        m, shape = _layer(ft, name)
        x = torch.randn(shape[0], cin, *shape[2:], device="cuda")
        for dtype, autocast in ((torch.float32, True), (torch.bfloat16, False)):
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast), pytest.raises(RuntimeError):
                m(x.to(dtype))


def test_fp32_without_autocast_selects_todays_functions(ft):
    for name, want in [("linear", "LinearCFBackward"), ("down-k2s2", "LinearCFBackward"), ("up-k2s2", "LinearCFBackward"),
                       ("head-k1", "LinearCFBackward"), ("stem", "ConvWgradCFBackward")]:
        m, shape = _layer(ft, name)
        shape = (2, 4, 16, 16, 32) if name == "stem" else shape       # the unfolded fp32 weight gradient needs 4096 voxels
        y = m(torch.randn(*shape, device="cuda"))
        names = _node_names(y)
        assert y.dtype == torch.float32 and any(want in n for n in names) and not any("Bf16" in n for n in names), (name, names)


def _stock(m, x):
    from factorizer_b200 import layers
    if isinstance(m, layers.ConvTranspose3d):
        return nn.ConvTranspose3d.forward(m, x)
    if isinstance(m, nn.modules.conv._ConvNd):
        return type(m).__mro__[2].forward(m, x)               # the nn.ConvNd under the mixin
    w = m.linear.weight.squeeze(-1)
    xf = x.flatten(2)
    y = torch.baddbmm(m.linear.bias[None, :, None], w.unsqueeze(0).expand(x.shape[0], -1, -1), xf)
    return y.view(x.shape[0], -1, *x.shape[2:])


def test_fp16_autocast_and_refused_shapes_match_the_stock_modules(ft):
    from factorizer_b200 import layers
    with torch.autocast("cuda", dtype=torch.float16):
        for name in LAYERS:
            m, shape = _layer(ft, name)
            x = torch.randn(*shape, device="cuda")
            y = m(x)
            assert y.dtype == torch.float16 and torch.equal(y, _stock(m, x)), name
    cases = []
    m, _ = _layer(ft, "linear")
    cases.append((m, torch.randn(1, 48, 5, 5, 5, device="cuda")))                   # 125 voxels
    m, _ = _layer(ft, "head-k1")
    base = torch.randn(32 * 16 ** 3 + 1, device="cuda").bfloat16()
    cases.append((m, base[1:].view(1, 32, 16, 16, 16)))                             # bf16, 2 bytes off a 16-byte boundary
    m, _ = _layer(ft, "down-k2s2")
    cases.append((m, torch.randn(1, 32, 6, 6, 12, device="cuda")))                  # 3 * 3 * 6 output voxels
    torch.manual_seed(8)
    cases.append((layers.Conv2d(16, 32, kernel_size=2, stride=2).cuda(), torch.randn(2, 16, 32, 32, device="cuda")))
    with torch.autocast("cuda", dtype=torch.bfloat16):
        for m, x in cases:
            y = m(x)
            assert not any("Bf16" in n for n in _node_names(y))
            assert torch.equal(y, _stock(m, x)), type(m).__name__


# ---- 4. whole model --------------------------------------------------------------------------------------------------------------
def _model(ft, dropout=0.1, n=128):
    torch.manual_seed(1234)
    return ft.Factorizer(in_channels=4, out_channels=3, spatial_size=(n, n, n), encoder_depth=(1, 1, 1, 1, 1),
                         encoder_width=(32, 64, 128, 256, 512), strides=(1, 2, 2, 2, 2), decoder_depth=(1, 1, 1, 1),
                         norm=ft.LayerNorm, reshape=(ft.SWMatricize, {"head_dim": 8, "patch_size": 8}), act=nn.ReLU,
                         factorize=ft.NMF, rank=1, num_iters=5, init="uniform", solver="hals", mlp_ratio=2, dropout=dropout).cuda()


def _library_scaffold(mp):
    from factorizer_b200 import _ops
    mp.setattr(_ops, "bf16_layer_supported", lambda *a, **k: False)


def _rel(a, ref):
    return float((a.double() - ref.double()).norm() / ref.double().norm().clamp_min(1e-300))


def test_swin_factorizer_bf16_scaffold_against_fp32(ft, monkeypatch):
    n = 128
    net = _model(ft)
    net.train()
    x = torch.rand(1, 4, n, n, n, device="cuda")
    target = torch.randint(0, 2, (1, 3, n, n, n), device="cuda").float()
    nodes = {}
    scaffold = [net.stem, net.head] + [lvl.downsample for lvl in net.encoder.blocks if not isinstance(lvl.downsample, nn.Identity)] \
        + [lvl.upsample for lvl in net.decoder.blocks] + [lvl.block.adapter for lvl in net.decoder.blocks]
    handles = [mod.register_forward_hook(lambda mod, inp, out: nodes.__setitem__(mod, _node_names(out))) for mod in scaffold]
    # under autocast the library keeps the head (3 outputs) and the 16^3 and 32^3 adapters (_ops.bf16_library_faster)
    library = {net.head} | {lvl.block.adapter for lvl in net.decoder.blocks if lvl.block.adapter.linear.in_channels >= 256}

    def step(autocast):
        net.zero_grad(set_to_none=True)
        nodes.clear()
        torch.manual_seed(77)
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
    for mod in scaffold:
        assert any(k in ROUTE for k in nodes[mod]) == (mod not in library), (type(mod).__name__, nodes[mod])
    with monkeypatch.context() as mp:
        _library_scaffold(mp)
        old = step(True)
        assert not any(k in ROUTE for mod in scaffold for k in nodes[mod])
    for h in handles:
        h.remove()
    names = ["loss"] + [k for k, _ in net.named_parameters()]
    for name, a, o, t in zip(names, [new[0]] + new[1], [old[0]] + old[1], [truth[0]] + truth[1]):
        if float(t.double().norm()) == 0.0:
            continue
        en, eo = _rel(a, t), _rel(o, t)
        print(f"model {name}: new scaffold {en:.3g}, library scaffold {eo:.3g}")
        assert en <= max(1.5 * eo, 2e-3), f"{name}: relative error {en:.3g} > max(1.5 x {eo:.3g}, 2e-3)"


# generic ATen kernels (by template name) and library GEMM / convolution kernels (by vendor name)
GENERIC = ("CatArrayBatchedCopy", "elementwise_kernel", "reduce_kernel", "fused_dropout", "bernoulli", "fill_kernel")
LIBRARY = ("cudnn", "cublas", "cutlass", "gemm", "nvjet", "xmma", "sm100_", "sm90_", "convolve", "wgrad", "dgrad", "fprop")


def _kernels(prof):
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
            and "memset" not in e.name.lower() and "memcpy" not in e.name.lower()]


# scaffold layers at the README model's shapes on the bf16 route, and the non-fz kernels each may launch forward + backward:
# the up-sampler's bias repeated per (co, k) and the sum of its gradient, and the copy of its weight gradient into the
# (ci, co, k) layout of the parameter -- all parameter-sized
def _scaffold_at_model_shapes(ft):
    from factorizer_b200 import layers
    bf = torch.bfloat16
    return {
        "stem": (layers.Conv3d(4, 32, kernel_size=3, padding=1, bias=False), (1, 4, 128, 128, 128), torch.float32, 0),
        "down 32->64": (layers.Conv3d(32, 64, kernel_size=2, stride=2), (1, 32, 128, 128, 128), bf, 0),
        "up 64->32": (layers.ConvTranspose3d(64, 32, kernel_size=2, stride=2), (1, 64, 64, 64, 64), bf, 3),
        "adapter 64->32": (ft.Linear(64, 32, bias=False), (1, 64, 128, 128, 128), bf, 0),
    }


def test_scaffold_layers_run_only_library_kernels(ft):
    """Forward + backward of each scaffold layer on the bf16 route launches this library's kernels and nothing else but the
    parameter-sized ops listed above: an unfold, a permutation copy or a dtype conversion of an activation would show here."""
    from torch.profiler import ProfilerActivity, profile
    torch.manual_seed(12)
    bad = {}
    for name, (m, shape, dtype, allowed) in _scaffold_at_model_shapes(ft).items():
        m = m.cuda()
        x = torch.randn(*shape, device="cuda").to(dtype).requires_grad_(name != "stem")
        gy = None

        def step():
            nonlocal gy
            m.zero_grad(set_to_none=True)                   # gradients are written, not accumulated
            x.grad = None
            with torch.autocast("cuda", dtype=torch.bfloat16):
                y = m(x)
            gy = torch.randn_like(y) if gy is None else gy
            y.backward(gy)
            return y

        assert any(k in ROUTE for k in _node_names(step())), name
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step()
            torch.cuda.synchronize()
        others = [k for k in _kernels(prof) if "fz::" not in k]
        print(name, len(others), others)
        bad.update({name: others} if len(others) > allowed or not all(any(g in k for g in GENERIC) for k in others) else {})
    assert not bad, bad


def test_swin_factorizer_bf16_step_kernels(ft):
    """The model's bf16 autocast step: library GEMMs and convolutions run only where the speed rule chose them (the head's
    3-output convolution; Linear over fewer than 65536 voxels: the 16^3 and 32^3 adapters and the 8^3 bottleneck block's
    layers), no unfold or padding op runs, and every other kernel is this library's or a generic ATen one (the skip `cat`,
    the positional-embedding add and dropout, the bottleneck block's elementwise ops and dtype conversions, parameter-sized
    ops)."""
    net = _model(ft)
    net.train()
    x = torch.rand(1, 4, 128, 128, 128, device="cuda")

    def step():
        net.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            logits = net(x)
        logits.backward(torch.ones_like(logits))

    step()
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA], record_shapes=True) as prof:
        step()
        torch.cuda.synchronize()
    ops = [(e.name, [list(sh) for sh in e.input_shapes if sh]) for e in prof.events()
           if e.device_type == torch.autograd.DeviceType.CPU and e.name.startswith("aten::")]
    names = {n for n, _ in ops}
    assert not names & {"aten::im2col", "aten::col2im", "aten::unfold", "aten::constant_pad_nd", "aten::stack"}, names
    for n, shapes in ops:
        if n in ("aten::cudnn_convolution", "aten::convolution_backward", "aten::_convolution"):
            assert [3, 32, 1, 1, 1] in shapes, (n, shapes)                                 # the head
        if n in ("aten::bmm", "aten::baddbmm", "aten::mm", "aten::addmm"):
            assert max(d for sh in shapes for d in sh) < 65536, (n, shapes)             # a Linear below 65536 voxels
    kernels = _kernels(prof)
    others = sorted({k for k in kernels if "fz::" not in k})
    print("\n".join(others))
    assert all(any(a in k for a in GENERIC) or any(s in k.lower() for s in LIBRARY) for k in others), others
    for fn in ("stem_wgrad_bf16_tc", "conv3_stem_fwd", "space_depth2", "linear_fwd_bf16_tc", "linear_wgrad_bf16_tc"):
        assert any(fn in k for k in kernels), fn


def test_swin_factorizer_bf16_step_cuda_graph_replays_eager(ft):
    net = _model(ft, dropout=0.0)
    net.train()
    x = torch.rand(1, 4, 128, 128, 128, device="cuda")
    params = list(net.parameters())
    static = {}

    def step():
        with torch.autocast("cuda", dtype=torch.bfloat16, cache_enabled=False):      # no cached casts across the capture
            logits = net(x)
        logits.float().square().mean().backward()
        return logits

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            net.zero_grad(set_to_none=True)
            step()
        net.zero_grad(set_to_none=True)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            static["logits"] = step()
    torch.cuda.current_stream().wait_stream(side)
    g.replay()
    torch.cuda.synchronize()
    grads = lambda: [torch.zeros_like(p) if p.grad is None else p.grad.clone() for p in params]
    got = [static["logits"].clone()] + grads()
    net.zero_grad(set_to_none=True)
    want = [step()] + grads()
    assert torch.equal(got[0], want[0])
    # the parameter gradients are sums over CTAs added with atomics, whose order is not fixed
    for a, b in zip(got[1:], want[1:]):
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-6 * float(b.abs().max()))
