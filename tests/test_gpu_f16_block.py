"""FactorizerBlock on fp16 activations (torch.autocast("cuda")'s default dtype, MONAI's amp): the fp16 instantiations of the
channel maps, weight gradient and weight staging (csrc/fz_bf16_block.cu), of the LayerNorm (csrc/fz_layernorm.cu) and of the
fused core (octant, paired and sub-warp kernels); _ops.FactorizerBlockF16Fn.

1. The kernels through the C ABI against fp64 on fp16-representable inputs: the channel map (every epilogue, with and without
   bias, both pipeline depths, partial tiles, 4 to 512 channels) to |y - ref| <= 2^-11 |ref| + TAU S, the weight gradient at
   production reduction lengths to TAU S, the LayerNorm forward and backward to one fp16 rounding, the staged weights equal
   to w.half() and its transpose with zero padding, a sum beyond 65504 stored as +-inf, and the bf16 entries' refusals.
2. The core at paths 2 (octant), 4 (paired window sets) and 3 (sub-warp) against the fp32 kernels on x.float(): bit for bit
   after one rounding on the sub-warp kernels (as the bf16 tests assert there), within one fp16 ulp on the octant paths.
3. The block against the fp32 block on x.float(): the relative Frobenius error of out, dx and every parameter gradient is at
   most max(1.5 x that of the fp16 autocast route without these kernels -- layer by layer, the core cast to fp32 -- , 2e-3);
   its node, its kernels, its saved memory, CUDA-graph replay, and the inputs it leaves to the layer-by-layer route.
4. Two models under torch.autocast("cuda") with torch.amp.GradScaler: loss and unscaled gradients against fp32 under the
   same rule, and an overflowing scale skips the step.
"""
import math

import numpy as np
import pytest
import torch
from torch import nn

pytestmark = pytest.mark.gpu

TAU = 2e-5
F = torch.nn.functional
EPI_NONE, EPI_RESIDUAL, EPI_GELU, EPI_GELU_GRAD, EPI_GELU_ONLY = 0, 1, 2, 3, 4
ISLES_RESHAPE = dict(head_dim=8, patch_size=4, shifts=[None, 1, 2, 3])


@pytest.fixture(scope="module")
def ft():
    from factorizer_b200 import _build
    _build.build()
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


def _h(*shape, scale=1.0, positive=False):
    t = torch.rand(*shape, device="cuda") if positive else torch.randn(*shape, device="cuda")
    return (scale * t).half()


def _gelu64(h):
    return 0.5 * h * (1.0 + torch.erf(h / math.sqrt(2.0)))


def _gelu_grad64(h):
    return 0.5 * (1.0 + torch.erf(h / math.sqrt(2.0))) + h * torch.exp(-0.5 * h * h) / math.sqrt(2.0 * math.pi)


def _ld8(n):
    return (n + 7) // 8 * 8


def _assert_bound(got, ref, S, what, rel=2.0 ** -11):
    err = (got.double() - ref).abs()
    excess = float((err - rel * ref.abs() - TAU * S).max())
    worst = float((err / (rel * ref.abs() + TAU * S).clamp_min(1e-300)).max())
    print(f"{what}: max err / (2^-11 |ref| + TAU S) = {worst:.3g}")
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
def test_channel_map_f16_against_fp64(lib, sms, name):
    B, cin, cout, vox, regime = CHANNEL_MAP_CASES[name]
    assert _fwd_regime(sms, B, cout, cin, vox) == regime or sms != 148
    torch.manual_seed(11)
    x = _h(B, cin, vox)
    w = _h(cout, cin, scale=1.0 / math.sqrt(cin))
    wpad = torch.zeros(cout, _ld8(cin), device="cuda", dtype=torch.float16)
    wpad[:, :cin] = w
    bias = 0.3 * torch.randn(cout, device="cuda")
    aux = _h(B, cout, vox)
    x64, w64, a64 = x.double(), w.double(), aux.double()
    r = torch.einsum("oc,bcv->bov", w64, x64)
    S = torch.einsum("oc,bcv->bov", w64.abs(), x64.abs())
    for epi in (EPI_NONE, EPI_RESIDUAL, EPI_GELU, EPI_GELU_GRAD, EPI_GELU_ONLY):
        for b in (bias, None):
            rb = r if b is None else r + b.double()[None, :, None]
            Sb = S if b is None else S + b.double().abs()[None, :, None]
            y = torch.full((B, cout, vox), float("nan"), device="cuda", dtype=torch.float16)
            y2 = torch.full_like(y, float("nan")) if epi == EPI_GELU else None
            use_aux = aux if epi in (EPI_RESIDUAL, EPI_GELU_GRAD) else None
            _check(lib.fz_linear_forward_f16(_p(x), _p(wpad), _ld8(cin), _p(b), _p(y), B, cin, cout, vox, epi, _p(use_aux), _p(y2),
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


def test_channel_map_f16_overflow_is_inf(lib):
    """a sum beyond the fp16 range is stored as +-inf (round to nearest), not clamped to 65504: GradScaler must see it"""
    B, cin, cout, vox = 1, 64, 64, 256
    x = torch.full((B, cin, vox), 64.0, device="cuda", dtype=torch.float16)
    w = torch.full((cout, cin), 32.0, device="cuda", dtype=torch.float16)
    w[cout // 2:] = -32.0                                     # 64 x 64 x 32 = 131072 > 65504
    y = torch.zeros(B, cout, vox, device="cuda", dtype=torch.float16)
    _check(lib.fz_linear_forward_f16(_p(x), _p(w), cin, None, _p(y), B, cin, cout, vox, EPI_NONE, None, None, _st()))
    assert bool((y[:, :cout // 2] == float("inf")).all()) and bool((y[:, cout // 2:] == float("-inf")).all())
    # just inside the range: 65504 itself is finite
    w = torch.full((cout, cin), 65504.0 / (64 * 64), device="cuda", dtype=torch.float16)
    ref = float((torch.full((cin,), 64.0, dtype=torch.float64) * float(w[0, 0])).sum())
    _check(lib.fz_linear_forward_f16(_p(x), _p(w), cin, None, _p(y), B, cin, cout, vox, EPI_NONE, None, None, _st()))
    assert bool(torch.isfinite(y).all()) and float(y.double().sub(ref).abs().max()) <= 2.0 ** -11 * ref


def test_channel_map_f16_refuses_what_it_cannot_read(lib):
    x = torch.zeros(1, 16, 64 + 8, device="cuda", dtype=torch.float16)
    w = torch.zeros(16, 16, device="cuda", dtype=torch.float16)
    y = torch.zeros(1, 16, 64, device="cuda", dtype=torch.float16)
    from factorizer_b200 import _lib as L
    assert lib.fz_linear_forward_f16(_p(x) + 2, _p(w), 16, None, _p(y), 1, 16, 16, 64, 0, None, None, _st()) == L.FZ_ERR_UNSUPPORTED
    assert lib.fz_linear_forward_f16(_p(x), _p(w), 16, None, _p(y), 1, 16, 16, 60, 0, None, None, _st()) == L.FZ_ERR_UNSUPPORTED
    assert lib.fz_linear_forward_f16(_p(x), _p(w), 12, None, _p(y), 1, 12, 16, 64, 0, None, None, _st()) == L.FZ_ERR_UNSUPPORTED
    assert lib.fz_linear_forward_f16(_p(x), _p(w), 16, None, _p(y) + 1, 1, 16, 16, 64, 0, None, None, _st()) == L.FZ_ERR_UNSUPPORTED
    dw = torch.zeros(16, 16, device="cuda")
    assert lib.fz_linear_wgrad_f16(_p(x) + 2, _p(x), _p(dw), None, 1, 16, 16, 64, _st()) == L.FZ_ERR_UNSUPPORTED
    assert lib.fz_linear_wgrad_f16(_p(x), _p(x), _p(dw), None, 1, 16, 16, 60, _st()) == L.FZ_ERR_UNSUPPORTED
    assert not lib.fz_linear_forward_f16_supported(16, 16, 60) and lib.fz_linear_forward_f16_supported(4, 4, 8)
    assert not lib.fz_linear_wgrad_f16_supported(16, 16, 60) and lib.fz_linear_wgrad_f16_supported(4, 4, 8)
    buf = torch.zeros(1024, device="cuda", dtype=torch.float16)
    w32 = torch.zeros(16, 16, device="cuda")
    assert lib.fz_f16_stage_weight(_p(w32), 16, 16, _p(buf) + 2, _st()) == L.FZ_ERR_UNSUPPORTED


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
def test_weight_gradient_f16_against_fp64(lib, name, data):
    B, cout, cin, vox = WGRAD_CASES[name]
    torch.manual_seed(5)
    pos = data == "same-sign"
    dy, x = _h(B, cout, vox, positive=pos), _h(B, cin, vox, positive=pos)
    dw = torch.full((cout, cin), float("nan"), device="cuda")
    db = torch.full((cout,), float("nan"), device="cuda")
    _check(lib.fz_linear_wgrad_f16(_p(dy), _p(x), _p(dw), _p(db), B, cout, cin, vox, _st()))
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


# ---- 1c. LayerNorm, staging ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,B,vox", [(32, 2, 32 ** 3), (64, 1, 64 ** 3), (64, 2, 4096), (128, 1, 32 ** 3), (256, 1, 4096),
                                     (512, 1, 4096), (100, 1, 1000)])
def test_layernorm_f16_against_fp64(lib, C, B, vox):
    torch.manual_seed(7)
    eps = 1e-5
    x = (_h(B, C, vox, scale=2.0) + 0.5).half()
    g, b = 1 + 0.3 * torch.randn(C, device="cuda"), 0.3 * torch.randn(C, device="cuda")
    y = torch.empty_like(x)
    _check(lib.fz_layernorm_cf_forward_f16(_p(x), _p(g), _p(b), _p(y), B, C, vox, eps, _st()))
    xd = x.double().requires_grad_(True)
    gd, bd = g.double().requires_grad_(True), b.double().requires_grad_(True)
    yd = F.layer_norm(xd.movedim(1, -1), (C,), gd, bd, eps).movedim(-1, 1)
    xhat = F.layer_norm(x.double().movedim(1, -1), (C,), None, None, eps).movedim(-1, 1)
    scale = (g.double().abs()[None, :, None] * xhat.abs() + b.double().abs()[None, :, None])
    err = (y.double() - yd).abs()
    # one fp16 rounding: half a unit in the last place, 2^-11 |y| for normal values and 2^-25 for subnormal ones
    worst = float((err / (2.0 ** -11 * yd.abs() + 2.0 ** -25 + 1e-5 * scale)).max())
    print(f"LN fwd C={C}: max err / (one fp16 rounding + 1e-5 scale) = {worst:.3g}")
    assert worst <= 1.0
    gy, add = _h(B, C, vox), _h(B, C, vox)
    dx = torch.empty_like(x)
    dg, db = torch.empty_like(g), torch.empty_like(b)
    _check(lib.fz_layernorm_cf_backward_add_f16(_p(x), _p(g), _p(gy), _p(add), _p(dx), _p(dg), _p(db), B, C, vox, eps, _st()))
    rx, rg, rb = torch.autograd.grad((yd * gy.double()).sum(), [xd, gd, bd])
    rx = rx + add.double()
    errx = float(((dx.double() - rx).abs() / (2.0 ** -11 * rx.abs() + 1e-5 * float(rx.abs().max()))).max())
    Sg = (gy.double().abs() * xhat.abs()).sum((0, 2))
    Sb = gy.double().abs().sum((0, 2))
    errg = float(((dg.double() - rg).abs() / Sg).max())
    errb = float(((db.double() - rb).abs() / Sb).max())
    print(f"LN bwd C={C}: dx {errx:.3g}, d(gamma) err/S {errg:.3g}, d(beta) err/S {errb:.3g}")
    assert errx <= 1.0 and errg <= 1e-5 and errb <= 1e-5
    assert lib.fz_layernorm_cf_f16_supported(C, vox) and not lib.fz_layernorm_cf_f16_supported(C, 1001)


def test_weight_staging_f16(ft, lib):
    from factorizer_b200 import _ops
    torch.manual_seed(1)
    shapes = [(64, 60), (60, 64), (128, 33), (7, 128)]
    ws = [torch.randn(*s, device="cuda") for s in shapes]
    buf = _ops._stage_weights_bf16(*ws, dtype=torch.float16)
    assert buf.dtype == torch.float16
    assert buf.numel() == sum(int(lib.fz_f16_staged_elems(*s)) for s in shapes)
    for w, ((a, lda), (at, ldt)) in zip(ws, _ops._staged_views(buf, shapes)):
        R, C = w.shape
        a, at = a.view(R, lda), at.view(C, ldt)
        assert torch.equal(a[:, :C], w.half()) and torch.equal(at[:, :R], w.t().half())
        assert not bool(a[:, C:].any()) and not bool(at[:, R:].any())
    one = _ops._stage_weights_bf16(ws[2], dtype=torch.float16)
    (a, lda), (at, ldt) = _ops._staged_views(one, [shapes[2]])[0]
    assert torch.equal(a.view(128, lda)[:, :33], ws[2].half()) and torch.equal(at.view(33, ldt)[:, :128], ws[2].t().half())


# ---- 2. the core --------------------------------------------------------------------------------------------------------------
CORE_CASES = {
    # name: (x shape, reshape kwargs, expected fz_last_path)
    "octant-[None,4]": ((2, 32, 32, 32, 32), dict(head_dim=8, patch_size=8), 2),
    "paired-[None,2,4,6]": ((1, 16, 32, 32, 32), dict(head_dim=8, patch_size=8, shifts=[None, 2, 4, 6]), 4),
    "sub-warp-isles22": ((2, 32, 32, 32, 32), ISLES_RESHAPE, 3),
}


def _ulp16(v):
    """the fp16 spacing at |v| (subnormal spacing below 2^-14)"""
    e = torch.floor(torch.log2(v.double().abs().clamp_min(2.0 ** -14)))
    return torch.exp2(e - 10)


@pytest.mark.parametrize("name", list(CORE_CASES))
def test_core_f16_against_fp32_kernels(ft, name):
    from factorizer_b200 import _lib, _ops
    xs, kw, path = CORE_CASES[name]
    rng = np.random.default_rng(40)
    r = ft.SWMatricize((None, *xs[1:]), **kw)
    M, N = r.output_size[2:]
    torch.manual_seed(3)
    nmf = ft.NMF((M, N), rank=1, num_iters=5, init="uniform", solver="hals").cuda()
    assert _ops.f16_core_supported(r._geom, nmf.solver_spec())
    x = torch.from_numpy(rng.standard_normal(xs).astype(np.float32)).cuda().half()
    gy = torch.from_numpy(rng.standard_normal(xs).astype(np.float32)).cuda().half()

    def run(v):
        v = v.clone().requires_grad_(True)
        y = _ops.SWNMF.apply(v, nmf.init.u0, nmf.init.v0, r._geom, nmf.solver_spec(), True)
        assert _lib.lib().fz_last_path() == path
        (gx,) = torch.autograd.grad(y, v, gy.to(v.dtype))
        assert _lib.lib().fz_last_path() == path
        return y.detach(), gx

    y, gx = run(x)
    assert y.dtype == torch.float16 and gx.dtype == torch.float16
    y32, gx32 = run(x.float())
    for what, a, t in (("y", y, y32), ("dx", gx, gx32)):
        assert bool(torch.isfinite(a).all()), what
        bitwise = torch.equal(a, t.half())
        worst = float(((a.double() - t.double()).abs() / _ulp16(t)).max())
        print(f"{name} {what}: bit for bit after one rounding: {bitwise}; max |fp16 - fp32| = {worst:.3g} fp16 ulp")
        if path == 3:                      # the sub-warp kernels: the fp32 kernels' sums, rounded once
            assert bitwise, what
        else:
            assert worst <= 1.0, what


def test_core_f16_refuses_one_patch_along_w(ft):
    from factorizer_b200 import _ops
    r = ft.SWMatricize((None, 64, 8, 8, 8), head_dim=8, patch_size=8)
    nmf = ft.NMF(r.output_size[2:], rank=1, num_iters=5, init="uniform", solver="hals").cuda()
    assert not _ops.f16_core_supported(r._geom, nmf.solver_spec())
    x = torch.rand(1, 64, 8, 8, 8, device="cuda").half()
    with pytest.raises(NotImplementedError, match="bf16 and fp16 volumes"):
        _ops.SWNMF.apply(x, nmf.init.u0, nmf.init.v0, r._geom, nmf.solver_spec(), True)


# ---- 3. the block ----------------------------------------------------------------------------------------------------------------
def _block(ft, C, n, ratio=2, reshape=None, seed=3):
    torch.manual_seed(seed)
    blk = ft.FactorizerBlock(channels=C, spatial_size=(n, n, n), norm=ft.LayerNorm,
                             reshape=(ft.SWMatricize, reshape or {"head_dim": 8, "patch_size": 8}), act=nn.ReLU, factorize=ft.NMF,
                             rank=1, num_iters=5, init="uniform", solver="hals", mlp_ratio=ratio, dropout=0.0).cuda()
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


def _old_route(mp):
    """fp16 autocast without these kernels: the layers one by one, FactMixer casting the core's input to fp32"""
    from factorizer_b200 import _ops
    mp.setattr(_ops, "f16_block_supported", lambda *a, **k: False)
    mp.setattr(_ops, "f16_core_supported", lambda *a, **k: False)


def _rel(a, ref):
    return float((a.double() - ref.double()).norm() / ref.double().norm().clamp_min(1e-300))


BLOCK_CASES = {
    # name: (C, B, n, ratio, reshape)
    "32ch-32^3": (32, 1, 32, 2, None),
    "64ch-2x32^3-ratio4": (64, 2, 32, 4, None),
    "128ch-16^3": (128, 1, 16, 2, None),
    "256ch-16^3-ratio4": (256, 1, 16, 4, None),
    "512ch-16^3": (512, 1, 16, 2, None),
    "64ch-paired-[None,2,4,6]": (64, 1, 32, 2, dict(head_dim=8, patch_size=8, shifts=[None, 2, 4, 6])),
    "64ch-isles22": (64, 2, 32, 2, ISLES_RESHAPE),
}


@pytest.mark.parametrize("name", list(BLOCK_CASES))
def test_block_f16_against_fp32(ft, monkeypatch, name):
    C, B, n, ratio, reshape = BLOCK_CASES[name]
    blk = _block(ft, C, n, ratio, reshape)
    torch.manual_seed(9)
    x = torch.randn(B, C, n, n, n, device="cuda").half()
    gout = torch.randn(B, C, n, n, n, device="cuda").half()
    out_t, grads_t, fn_t = _run(blk, x.float(), gout.float())                 # fp32 truth (fused fp32 path)
    assert type(fn_t).__name__ in ("FactorizerBlockFnBackward", "FactorizerBlockWideFnBackward")
    out_n, grads_n, fn_n = _run(blk, x, gout)                                 # fp16 input, no autocast
    assert type(fn_n).__name__ == "FactorizerBlockF16FnBackward"
    assert out_n.dtype == torch.float16 and grads_n[0].dtype == torch.float16
    assert all(g.dtype == torch.float32 for g in grads_n[1:])
    with torch.autocast("cuda"):                                              # fp16 autocast: the same node
        out_a, _, fn_a = _run(blk, x, gout)
    assert type(fn_a).__name__ == "FactorizerBlockF16FnBackward" and torch.equal(out_a, out_n)
    with monkeypatch.context() as mp:                                         # the fp16 route without these kernels
        _old_route(mp)
        with torch.autocast("cuda"):
            out_o, grads_o, fn_o = _run(blk, x, gout)
    assert type(fn_o).__name__ != "FactorizerBlockF16FnBackward"
    names = ["out", "dx"] + [k for k, _ in blk.named_parameters()]
    for pname, a, o, t in zip(names, [out_n] + grads_n, [out_o] + grads_o, [out_t] + grads_t):
        en, eo = _rel(a, t), _rel(o, t)
        bound = max(1.5 * eo, 2e-3)
        print(f"{name} {pname}: fp16 block {en:.3g}, fp16 layer by layer {eo:.3g}")
        assert en <= bound, f"{pname}: relative error {en:.3g} > max(1.5 x {eo:.3g}, 2e-3)"


def test_block_f16_runs_only_library_kernels(ft):
    blk = _block(ft, 64, 32)
    x = torch.randn(1, 64, 32, 32, 32, device="cuda").half().requires_grad_(True)
    gout = torch.randn(1, 64, 32, 32, 32, device="cuda").half()
    blk(x).backward(gout)
    blk.zero_grad(set_to_none=True)
    x.grad = None
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = blk(x)
        out.backward(gout)
        torch.cuda.synchronize()
    assert type(out.grad_fn).__name__ == "FactorizerBlockF16FnBackward"
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    kernels = {n for n in names if "memset" not in n.lower()}
    print(sorted(names))
    assert kernels and all("fz::" in n for n in kernels), sorted(n for n in kernels if "fz::" not in n)
    assert all("__half" in n for n in kernels if "linear_fwd_bf16_tc" in n or "linear_wgrad_bf16_tc" in n)
    assert any("linear_fwd_bf16_tc<__half" in n for n in kernels) and any("linear_wgrad_bf16_tc<__half" in n for n in kernels)
    assert any("phase_fwd_gram<__half" in n for n in kernels) and any("layernorm" in n and "__half" in n for n in kernels)


@pytest.mark.parametrize("C,n", [(64, 32), (128, 32), (256, 32)])
def test_block_f16_saves_half_the_memory(ft, C, n):
    blk = _block(ft, C, n)
    x32 = torch.randn(1, C, n, n, n, device="cuda").requires_grad_(True)
    x16 = x32.detach().half().requires_grad_(True)

    def growth(x):
        blk(x).float().sum().backward()                          # workspaces exist
        blk.zero_grad(set_to_none=True)
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        out = blk(x)
        torch.cuda.synchronize()
        grow = torch.cuda.memory_allocated() - before
        del out
        return grow

    g32, g16 = growth(x32), growth(x16)
    print(f"C={C} n={n}: forward keeps {g16} bytes in fp16, {g32} in fp32: {g16 / g32:.3f}")
    assert g16 <= 0.55 * g32


def test_block_f16_cuda_graph_replays_eager(ft):
    blk = _block(ft, 64, 32)
    x = torch.randn(2, 64, 32, 32, 32, device="cuda").half().requires_grad_(True)
    gout = torch.randn(2, 64, 32, 32, 32, device="cuda").half()
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
    assert type(out_g.grad_fn).__name__ == "FactorizerBlockF16FnBackward"
    blk.zero_grad(set_to_none=True)
    x.grad = None
    out = blk(x)
    out.backward(gout)
    want = [out, x.grad] + [p.grad for p in params]
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    # the parameter gradients are sums over CTAs added with atomics, whose order is not fixed
    for a, b in zip(got[2:], want[2:]):
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-6 * float(b.abs().max()))


def test_refused_f16_inputs_run_layer_by_layer(ft, monkeypatch):
    """what FactorizerBlockF16Fn does not take runs the layers one by one without raising, exactly as without it"""
    def both(blk, x):
        outs = []
        for patched in (False, True):
            with monkeypatch.context() as mp:
                if patched:
                    _old_route(mp)
                with torch.autocast("cuda"):
                    out, grads, fn = _run(blk, x, torch.ones_like(x))
            outs.append((out, grads, type(fn).__name__))
        (a, ga, fa), (b, gb, fb) = outs
        assert fa == fb and fa != "FactorizerBlockF16FnBackward", (fa, fb)
        assert torch.equal(a, b)
        for p, q in zip(ga, gb):
            assert torch.allclose(p.float(), q.float(), rtol=1e-5, atol=1e-6 * float(q.float().abs().max())), "gradient differs"

    # a geometry the fp16 core refuses: one patch along W (the 8^3 bottleneck); FactMixer casts the core's input to fp32
    both(_block(ft, 64, 8), torch.randn(1, 64, 8, 8, 8, device="cuda").half())
    # an fp16 x 2 bytes off a 16-byte boundary
    blk = _block(ft, 64, 16)
    base = torch.randn(64 * 16 ** 3 + 1, device="cuda").half()
    xm = base[1:].view(1, 64, 16, 16, 16)
    assert xm.data_ptr() % 16 and not ft._ops.f16_block_supported(xm, 128)
    both(blk, xm)


# ---- 4. models under fp16 autocast with GradScaler -----------------------------------------------------------------------------
def _model_under_fp16_autocast(ft, monkeypatch, net, B, n, deepest):
    """Every block but the bottleneck at `deepest` takes FactorizerBlockF16Fn; loss and unscaled gradients against fp32 meet
    max(1.5 x the error of the fp16 layer-by-layer route with the core cast to fp32, 2e-3)."""
    net.train()
    torch.manual_seed(5)
    x = torch.rand(B, 4, n, n, n, device="cuda")
    target = torch.randint(0, 2, (B, 3, n, n, n), device="cuda").float()
    nodes = {}

    def hook(mod, inp, out):
        nodes[mod] = (tuple(inp[0].shape[2:]), type(out.grad_fn).__name__)

    blocks = [m for m in net.modules() if isinstance(m, ft.FactorizerBlock)]
    handles = [b.register_forward_hook(hook) for b in blocks]
    opt = torch.optim.SGD(net.parameters(), lr=0.01)

    def step(autocast):
        net.zero_grad(set_to_none=True)
        nodes.clear()
        torch.manual_seed(77)                     # the positional-embedding dropout draws the same masks in every run
        scaler = torch.amp.GradScaler("cuda", enabled=autocast)
        with torch.autocast("cuda", enabled=autocast):
            logits = net(x)
        logits = logits.float()
        p = torch.sigmoid(logits)
        dice = 1 - (2 * (p * target).sum((2, 3, 4)) + 1e-5) / (p.sum((2, 3, 4)) + target.sum((2, 3, 4)) + 1e-5)
        loss = F.binary_cross_entropy_with_logits(logits, target) + dice.mean()
        scaler.scale(loss).backward()
        if autocast:
            scaler.unscale_(opt)                 # the gradients in place, divided by the scale; no overflow at the default
            assert all(bool(torch.isfinite(q.grad).all()) for q in net.parameters() if q.grad is not None)
        return loss.detach(), [q.grad.detach().clone() if q.grad is not None else torch.zeros_like(q) for q in net.parameters()]

    truth = step(False)
    new = step(True)
    for b in blocks:
        size, fn = nodes[b]
        print(size, fn)
        if size != deepest:
            assert fn == "FactorizerBlockF16FnBackward", (size, fn)
    with monkeypatch.context() as mp:
        _old_route(mp)
        old = step(True)
    names = ["loss"] + [k for k, _ in net.named_parameters()]
    for name, a, o, t in zip(names, [new[0]] + new[1], [old[0]] + old[1], [truth[0]] + truth[1]):
        if float(t.double().norm()) == 0.0:
            continue
        en, eo = _rel(a, t), _rel(o, t)
        print(f"model {name}: fp16 blocks {en:.3g}, fp16 layer by layer {eo:.3g}")
        assert en <= max(1.5 * eo, 2e-3), f"{name}: relative error {en:.3g} > max(1.5 x {eo:.3g}, 2e-3)"

    # a scale that overflows fp16: the scaler finds inf, skips the step and backs the scale off
    before = [q.detach().clone() for q in net.parameters()]
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 60)
    net.zero_grad(set_to_none=True)
    with torch.autocast("cuda"):
        logits = net(x)
    loss = F.binary_cross_entropy_with_logits(logits.float(), target)
    scaler.scale(loss).backward()
    scaler.step(opt)
    scaler.update()
    for h in handles:
        h.remove()
    assert scaler.get_scale() < 2.0 ** 60
    assert all(torch.equal(a, b) for a, b in zip(before, net.parameters()))


def test_swin_factorizer_under_fp16_autocast_with_grad_scaler(ft, monkeypatch):
    n = 128
    torch.manual_seed(1234)
    net = ft.Factorizer(in_channels=4, out_channels=3, spatial_size=(n, n, n), encoder_depth=(1, 1, 1, 1, 1),
                        encoder_width=(32, 64, 128, 256, 512), strides=(1, 2, 2, 2, 2), decoder_depth=(1, 1, 1, 1),
                        norm=ft.LayerNorm, reshape=(ft.SWMatricize, {"head_dim": 8, "patch_size": 8}), act=nn.ReLU,
                        factorize=ft.NMF, rank=1, num_iters=5, init="uniform", solver="hals", mlp_ratio=2, dropout=0.1).cuda()
    _model_under_fp16_autocast(ft, monkeypatch, net, 1, n, (8, 8, 8))


def test_isles22_factorizer_under_fp16_autocast_with_grad_scaler(ft, monkeypatch):
    """the ISLES22 stand-in of test_gpu_bf16_small_windows.py: head_dim 8, patch 4, shifts [None, 1, 2, 3], batch 8, 64^3"""
    n = 64
    torch.manual_seed(1234)
    net = ft.Factorizer(in_channels=4, out_channels=3, spatial_size=(n, n, n), encoder_depth=(1, 1, 1, 1, 1),
                        encoder_width=(32, 64, 128, 256, 512), strides=(1, 2, 2, 2, 2), decoder_depth=(1, 1, 1, 1),
                        norm=ft.LayerNorm, reshape=(ft.SWMatricize, ISLES_RESHAPE), act=nn.ReLU, factorize=ft.NMF, rank=1,
                        num_iters=5, init="uniform", solver="hals", dropout=0.1).cuda()
    _model_under_fp16_autocast(ft, monkeypatch, net, 8, n, (4, 4, 4))
