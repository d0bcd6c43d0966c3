"""The channel-map kernels at the shapes the Swin Factorizer runs them at, against fp64 torch on the device.

- fz_linear_forward_ex (csrc/fz_linear_tc.cu) with enough (voxel tile, output tile) items that persistent CTAs walk two
  to 28 of them: the running sums of an item are started (bias / residual) while the previous one drains, and the TMEM
  accumulator pair is reused across items; on either side of the 4-stage / 2-stage switch.
- fz_linear_wgrad on tcgen05 (glue mode 7) and on the FP32 pipe (mode 5) over production reduction lengths, where the
  launcher caps the tensor-core accumulation chain, on zero-mean and on same-sign operands.
- fz_mlp_backward / fz_linear_backward (the 32-channel block glue) beyond their tile-per-CTA caps, on operands with a
  positive mean.
- Buffers at a 4-byte offset: the C entry points that move 16-byte words refuse them, the layers fall back to torch.

Weight gradients are held to two bounds.  Condition-aware: |dW - dW64| <= TAU * S per entry, S the same contraction over
absolute values (the size of the sum the kernel actually forms; the error of a truncating accumulation chain scales with
S, not with the result, which cancels for zero-mean data).  And the bound of the other parity tests: scaled by
max(1, max|ref|), rtol = atol = 1e-4.  The shapes follow from the SM count, and each test asserts the launch regime it
is meant to exercise with the launcher's own formula.

Measured on a B200 (148 SMs, 1000 W power limit), max |err| / S:
    fz_linear_wgrad, tcgen05, chain capped at 32 stages   same-sign 7.7e-6 .. 1.04e-5 (capped shapes), 5.8e-6 (512 x 512
                                                          x 16^3, uncapped); zero-mean <= 2.4e-7.  With the former cap of
                                                          64 stages: 1.5e-5 .. 1.7e-5; without a cap: 9.8e-5 (443 stages)
    fz_linear_wgrad, FP32 pipe (all three kernels)        same-sign <= 1.0e-6; zero-mean <= 3.7e-8
    fz_mlp_backward, tcgen05 (192 tiles = 2304 MMAs)      dW1 1.35e-4, dW2 1.41e-4, d(gamma) 4.1e-5; the rest <= 1.9e-6
    fz_mlp_backward, FP32 pipe                            dW2 8.0e-6, the rest <= 1.5e-6
    fz_linear_backward, tcgen05 (111 tiles = 1776 MMAs)   dW_out 1.08e-4, dW_in 9.4e-5, d(gamma) 4.1e-5; the rest <= 7e-7
    fz_linear_backward, FP32 pipe                         <= 1.0e-6
With the 32-stage cap the worst linear_wgrad_tc case (64 -> 64 over 2 x 128^3) sits at 1.04e-5 S, 1.9x below TAU.  The glue
kernels' tensor-core chains lose about 2^-24 S per MMA, as linear_wgrad_tc did before its cap was lowered: their TAU check
is an expected failure (GLUE_CHECKS); the parity bound holds for them.
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

TAU = 2e-5
GUARD = 4096
SENTINEL = 12345.0
F = torch.nn.functional


@pytest.fixture(scope="module")
def lib():
    from factorizer_b200 import _lib as L
    return L.lib()


@pytest.fixture(scope="module")
def sms():
    assert torch.cuda.is_available()
    return torch.cuda.get_device_properties(0).multi_processor_count


def _check(code):
    from factorizer_b200 import _lib as L
    L.check(code)


def _st():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _tol_ratio(got, ref, rtol, atol):
    """max |got - ref| / (atol + rtol |ref|) over the device, in chunks; inf if anything is not finite"""
    g, r = got.reshape(-1), ref.reshape(-1)
    m = 0.0
    for i in range(0, g.numel(), 1 << 24):
        gc, rc = g[i:i + (1 << 24)].double(), r[i:i + (1 << 24)].double()
        if not bool(torch.isfinite(gc).all()):
            return math.inf
        m = max(m, float(((gc - rc).abs() / (atol + rtol * rc.abs())).max()))
    return m


def _grad_bounds(got, ref, S):
    """(max |got - ref| / S, the parity tests' ratio with the max(1, max|ref|) scaling at rtol = atol = 1e-4)"""
    if not bool(torch.isfinite(got).all()):
        return math.inf, math.inf
    err = (got.double() - ref).abs()
    scale = max(1.0, float(ref.abs().max()))
    return float((err / S.clamp_min(1e-300)).max()), float((err / scale / (1e-4 + 1e-4 * ref.abs() / scale)).max())


def _assert_grad(got, ref, S, what, with_tau=True):
    """with_tau=False: the parity bound alone (the ratio to S is still printed)"""
    cond, gate = _grad_bounds(got, ref, S)
    print(f"{what}: err/S = {cond:.3g}, parity ratio = {gate:.3g}")
    assert not with_tau or cond <= TAU, f"{what}: max |err| / S = {cond:.3g} > {TAU}"
    assert gate <= 1.0, f"{what}: max err / tol = {gate:.3g} (scaled by max(1, max|ref|), rtol = atol = 1e-4)"


def _gelu64(h):
    return 0.5 * h * (1.0 + torch.erf(h / math.sqrt(2.0)))


def _gelu_grad64(h):
    return 0.5 * (1.0 + torch.erf(h / math.sqrt(2.0))) + h * torch.exp(-0.5 * h * h) / math.sqrt(2.0 * math.pi)


class _Glue:
    """fz_set_glue_mode for the calling thread (the mode is thread-local), restored afterwards"""

    def __init__(self, lib, mode):
        self.lib, self.mode = lib, mode

    def __enter__(self):
        self.before = self.lib.fz_get_glue_mode()
        self.lib.fz_set_glue_mode(self.mode)

    def __exit__(self, *exc):
        self.lib.fz_set_glue_mode(self.before)


# ---- 1. fz_linear_forward_ex: items per CTA -----------------------------------------------------------------------------
def _fwd_regime(sms, B, cout, cin, vox):
    """linear_fwd_tc_launch: items, pipeline depth, CTAs, fewest / most items a CTA walks"""
    items = B * (-(-vox // 128)) * (-(-cout // 64))
    four = items <= sms and cin > 64
    ctas = items if four else min(items, 2 * sms)
    return items, four, items // ctas, -(-items // ctas)


def _fwd_case(sms, name):
    even = sms % 2 == 0
    if name == "one-item-4-stage":            # items == SMs, cin > 64
        B, vt = (2, sms // 2) if even else (1, sms)
        return B, 100, 64, vt * 128 - 4
    if name == "one-item-2-stage":            # items == SMs + 1
        return 1, 100, 64, sms * 128 + 124
    if name == "two-or-three-items":          # about 2.1 items per CTA, ragged tiles straddling samples
        return 2, 260, 136, round(0.7 * sms) * 128 - 56
    if name == "six-or-seven-items":          # (1, 512 -> 512): 6.5 items per CTA
        return 1, 512, 512, (13 * sms // 8) * 128
    if name == "partial-output-tile":         # cout = 3: every store predicated, 28 items per CTA
        return 2, 36, 3, 28 * sms * 128 - 12
    raise KeyError(name)


@pytest.mark.parametrize("name", ["one-item-4-stage", "one-item-2-stage", "two-or-three-items", "six-or-seven-items",
                                  "partial-output-tile"])
def test_channel_map_items_per_cta(lib, sms, name):
    """All five epilogues, with and without bias, the weight as stored and transposed (cout % 4 == 0), into NaN-filled
    outputs followed by a guard band; rtol 1e-4 / atol 1e-5 against the k=1 Conv1d of the reference in fp64."""
    B, cin, cout, vox = _fwd_case(sms, name)
    items, four, lo, hi = _fwd_regime(sms, B, cout, cin, vox)
    expect = {"one-item-4-stage": (items == sms and four and hi == 1),
              "one-item-2-stage": (items == sms + 1 and not four and hi == 1),
              "two-or-three-items": (not four and lo == 2 and hi == 3 and B >= 2 and vox % 128),
              "six-or-seven-items": (not four and lo == 6 and hi == 7),
              "partial-output-tile": (not four and lo >= 27 and cout % 64 and B >= 2 and vox % 128)}[name]
    assert expect, (name, items, four, lo, hi)
    torch.manual_seed(21)
    dev = torch.device("cuda:0")
    x = torch.randn(B, cin, vox, device=dev)
    W = torch.randn(cout, cin, device=dev) / cin ** 0.5
    bias = torch.randn(cout, device=dev)
    aux = torch.randn(B, cout, vox, device=dev)
    n = B * cout * vox
    ybuf = torch.empty(n + GUARD, device=dev)
    y2buf = torch.empty(n + GUARD, device=dev)
    ybuf[n:], y2buf[n:] = SENTINEL, SENTINEL
    y, y2 = ybuf[:n].view(B, cout, vox), y2buf[:n].view(B, cout, vox)
    r0 = torch.einsum("oc,bcv->bov", W.double(), x.double())
    gp = _gelu_grad64(aux.double())
    Wt = W.t().contiguous()
    bad = []
    for with_bias in (False, True):
        r = r0 + bias.double()[None, :, None] if with_bias else r0
        refs = {0: [r], 1: [r + aux.double()], 2: [r, _gelu64(r)], 3: [r * gp], 4: [_gelu64(r)]}
        for wt in ((0, 1) if cout % 4 == 0 else (0,)):
            for epi, ref in refs.items():
                y.fill_(float("nan"))
                y2.fill_(float("nan"))
                _check(lib.fz_linear_forward_ex(_p(x), _p(Wt if wt else W), _p(bias) if with_bias else None, _p(y), B, cin, cout,
                                                vox, epi, wt, _p(aux), _p(y2), _st()))
                for got, want, which in zip((y, y2), ref, ("y", "y2")):
                    q = _tol_ratio(got, want, 1e-4, 1e-5)
                    if q > 1.0:
                        bad.append(f"epilogue {epi} bias={with_bias} transposed={wt} {which}: max err / tol = {q:.3g}")
                for buf, which in ((ybuf, "y"), (y2buf, "y2")):
                    if not bool((buf[n:] == SENTINEL).all()):
                        bad.append(f"epilogue {epi} bias={with_bias} transposed={wt}: write past the end of {which}")
    assert not bad, "\n".join(bad)


# ---- 2. fz_linear_wgrad: production reduction lengths ---------------------------------------------------------------------
def _wgrad_tc_regime(sms, B, cout, cin, vox):
    """linear_wgrad_tc_launch: (stages per CTA without the cap, with it, whether the cap raised the grid)"""
    tiles = B * (-(-vox // 32))
    bo, bi = -(-cout // 64), -(-cin // 64)
    gx0 = min(max(-(-2 * sms // (bo * bi)), 1), tiles)
    gx = gx0
    if gx * 32 < tiles:
        gx = -(-tiles // 32)
    gx = min(max(gx, 1), tiles)
    return -(-tiles // gx0), -(-tiles // gx), gx != gx0


def _wgrad_fp32_kernel(B, cout, cin, vox):
    """the FP32-pipe kernel fz_linear_wgrad picks without the tensor cores"""
    if (cin >= 64 if cout >= 64 else cin > 64) and B * vox >= 32768:
        return "linear_wgrad64<2,1>" if cout >= 64 else "linear_wgrad64<1,2>"
    return "linear_wgrad"


# (B, cin, cout, vox), whether the tensor-core launch caps the chain
WGRAD_CASES = {"64-256-64^3": ((2, 64, 256, 64 ** 3), True), "64-64-128^3": ((2, 64, 64, 128 ** 3), True),
               "72-200-ragged": ((3, 72, 200, 40012), True), "512-512-16^3": ((1, 512, 512, 16 ** 3), False),
               "108-32-64^3": ((1, 108, 32, 64 ** 3), None), "40-24-30000": ((2, 40, 24, 30000), None)}


@pytest.mark.parametrize("data", ["zero-mean", "same-sign"])
@pytest.mark.parametrize("mode", [7, 5], ids=["tcgen05", "fp32-pipe"])
@pytest.mark.parametrize("name", list(WGRAD_CASES))
def test_linear_wgrad_long_reductions(lib, sms, name, mode, data):
    """dW = sum dy x^T and db = sum dy through the C ABI at glue mode 7 (tcgen05, 3xTF32, the chain capped at 32 stages of
    4 MMAs) and 5 (FP32 pipe), called from this thread (the mode is thread-local).  The last two shapes are the FP32-pipe
    kernels' other block shapes (32 x 128 for the stem's 108 unfolded rows, 32 x 32); the tensor cores take them too."""
    (B, cin, cout, vox), capped = WGRAD_CASES[name]
    if mode == 7 and capped is not None:
        uncapped, stages, engaged = _wgrad_tc_regime(sms, B, cout, cin, vox)
        assert engaged == capped and stages <= 32, (uncapped, stages, engaged)
    if mode == 5 and capped is None:
        assert _wgrad_fp32_kernel(B, cout, cin, vox) != "linear_wgrad64<2,1>"
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(31)
    dy = torch.randn(B, cout, vox, device=dev, generator=g)
    x = torch.randn(B, cin, vox, device=dev, generator=g)
    if data == "same-sign":
        dy.abs_().add_(0.1)
        x.abs_().add_(0.5)
    dW = torch.empty(cout, cin, device=dev)
    db = torch.empty(cout, device=dev)
    with _Glue(lib, mode):
        _check(lib.fz_linear_wgrad(_p(dy), _p(x), _p(dW), _p(db), B, cout, cin, vox, _st()))
    ref = torch.zeros(cout, cin, device=dev, dtype=torch.float64)
    S = torch.zeros_like(ref)
    for b in range(B):
        d64, x64 = dy[b].double(), x[b].double()
        ref += d64 @ x64.t()
        S += d64.abs() @ x64.abs().t()
        del d64, x64
    dbr, dbS = dy.double().sum((0, 2)), dy.double().abs().sum((0, 2))
    tag = f"{name} {'tcgen05' if mode == 7 else 'fp32-pipe'} {data}"
    _assert_grad(dW, ref, S, f"dW {tag}")
    _assert_grad(db, dbr, dbS, f"db {tag}")


# ---- 3. the 32-channel glue backward beyond its tile-per-CTA caps ------------------------------------------------------
def _glue_operands(B, C, hid, vox, seed):
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    r = lambda *s: torch.randn(*s, device=dev, generator=g)
    p = dict(x1=r(B, C, vox) + 2.0 * r(C)[None, :, None], m=r(B, C, vox).abs_(), dout=r(B, C, vox).abs_().add_(0.1),
             g=1 + 0.3 * r(C), b=0.3 * r(C), w1=r(hid, C) / 6, bb1=0.2 * r(hid), w2=r(C, hid) / 7, w=r(C, C) / 6)
    return p


def _chunks(B, vox, step=1 << 18):
    for b in range(B):
        for v0 in range(0, vox, step):
            yield b, slice(v0, min(vox, v0 + step))


def _ln64(x, eps):
    mu = x.mean(0, keepdim=True)
    rstd = ((x - mu).square().mean(0, keepdim=True) + eps).rsqrt()
    return (x - mu) * rstd, rstd


def _ln_back64(dxh, xh, rstd):
    return rstd * (dxh - dxh.mean(0, keepdim=True) - xh * (dxh * xh).mean(0, keepdim=True))


# mlp_bwd_tc and linear_bwd_tc2 accumulate their weight gradients in TMEM over every tile of a CTA (up to 192 tiles of 12
# MMAs, 128 tiles of 16 MMAs) and lose about 2^-24 S per MMA of that chain on same-sign data: 1.1e-4 .. 1.4e-4 S at these
# shapes, beyond TAU.  Their TAU check is an expected failure until the chains are cut (a periodic flush of the TMEM
# accumulator into registers, as linear_fwd_tc does per segment); the parity bound and the FP32-pipe kernels hold TAU.
_TC_CHAIN = ("mlp_bwd_tc / linear_bwd_tc2 accumulate the weight gradients over a CTA's whole chain of tiles in TMEM with "
             "truncation: 1.1e-4 .. 1.4e-4 S measured on a B200, TAU = 2e-5")
GLUE_CHECKS = [pytest.param(7, False, id="tcgen05-parity"),
               pytest.param(7, True, id="tcgen05-tau", marks=pytest.mark.xfail(strict=True, reason=_TC_CHAIN)),
               pytest.param(0, True, id="fp32-pipe")]


@pytest.mark.parametrize("mode,with_tau", GLUE_CHECKS)
@pytest.mark.parametrize("hid", [64, 128])
def test_mlp_backward_beyond_cap(lib, sms, hid, mode, with_tau):
    """fz_mlp_backward at (2, 32, 128^3): with the tensor cores more than 192 tiles of 96 voxels per SM, so the launcher adds
    CTAs.  Reference: the MLP half of the block written out in fp64, chunk by chunk over voxels.  The bounds S follow the
    kernel's factorisation dW1 = Q diag(gamma) + db1 beta^T with Q = sum dh xh^T (xh the normalised input), and
    d(gamma)_c = sum_j W1[j][c] Q[j][c], d(beta)_c = sum_j W1[j][c] db1[j]."""
    B, C, vox, eps = 2, 32, 128 ** 3, 1e-5
    tiles = B * (-(-vox // 96))
    nblk = max(min(tiles, sms), -(-tiles // 192))
    assert min(tiles, sms) * 192 < tiles and -(-tiles // nblk) == 192, "the 192-tile cap of mlp_bwd_tc is not engaged"
    p = _glue_operands(B, C, hid, vox, 41)
    dev = p["x1"].device
    got = dict(dx1=torch.empty(B, C, vox, device=dev), dg=torch.empty(C, device=dev), db=torch.empty(C, device=dev),
               dw1=torch.empty(hid, C, device=dev), dbb1=torch.empty(hid, device=dev), dw2=torch.empty(C, hid, device=dev),
               dbb2=torch.empty(C, device=dev))
    with _Glue(lib, mode):
        _check(lib.fz_mlp_backward(_p(p["x1"]), _p(p["dout"]), _p(p["g"]), _p(p["b"]), _p(p["w1"]), _p(p["bb1"]), _p(p["w2"]),
                                   *[_p(got[k]) for k in ("dx1", "dg", "db", "dw1", "dbb1", "dw2", "dbb2")], B, C, hid, vox, eps, _st()))
    d = lambda k: p[k].double()
    gm, bt, w1, bb1, w2 = d("g"), d("b"), d("w1"), d("bb1"), d("w2")
    z = lambda *s: torch.zeros(*s, device=dev, dtype=torch.float64)
    acc = dict(dw2=z(C, hid), S_dw2=z(C, hid), Q=z(hid, C), SQ=z(hid, C), dbb1=z(hid), S_dbb1=z(hid), dbb2=z(C), S_dbb2=z(C))
    dx1_ratio = 0.0
    for b, v in _chunks(B, vox):
        x1, dout = p["x1"][b, :, v].double(), p["dout"][b, :, v].double()
        xh, rstd = _ln64(x1, eps)
        h = w1 @ (gm[:, None] * xh + bt[:, None]) + bb1[:, None]
        g = _gelu64(h)
        dh = (w2.t() @ dout) * _gelu_grad64(h)
        del h
        acc["dw2"] += dout @ g.t()
        acc["S_dw2"] += dout.abs() @ g.abs().t()
        del g
        acc["Q"] += dh @ xh.t()
        acc["SQ"] += dh.abs() @ xh.abs().t()
        acc["dbb1"] += dh.sum(1)
        acc["S_dbb1"] += dh.abs().sum(1)
        acc["dbb2"] += dout.sum(1)
        acc["S_dbb2"] += dout.abs().sum(1)
        dx1 = dout + _ln_back64(gm[:, None] * (w1.t() @ dh), xh, rstd)
        dx1_ratio = max(dx1_ratio, _tol_ratio(got["dx1"][b, :, v], dx1, 1e-4, 2e-5))
        del dh, dx1, xh
    Q, SQ, aw1 = acc["Q"], acc["SQ"], w1.abs()
    tag = f"hidden {hid} {'tcgen05' if mode == 7 else 'fp32-pipe'}"
    _assert_grad(got["dw1"], Q * gm[None, :] + acc["dbb1"][:, None] * bt[None, :],
                 SQ * gm.abs()[None, :] + acc["S_dbb1"][:, None] * bt.abs()[None, :], f"dW1 {tag}", with_tau)
    _assert_grad(got["dbb1"], acc["dbb1"], acc["S_dbb1"], f"db1 {tag}", with_tau)
    _assert_grad(got["dw2"], acc["dw2"], acc["S_dw2"], f"dW2 {tag}", with_tau)
    _assert_grad(got["dbb2"], acc["dbb2"], acc["S_dbb2"], f"db2 {tag}", with_tau)
    _assert_grad(got["dg"], (w1 * Q).sum(0), (aw1 * SQ).sum(0), f"dgamma {tag}", with_tau)
    _assert_grad(got["db"], (w1 * acc["dbb1"][:, None]).sum(0), (aw1 * acc["S_dbb1"][:, None]).sum(0), f"dbeta {tag}", with_tau)
    assert dx1_ratio <= 1.0, f"dx1: max err / tol = {dx1_ratio:.3g} (rtol 1e-4, atol 2e-5)"


@pytest.mark.parametrize("mode,with_tau", GLUE_CHECKS)
@pytest.mark.parametrize("layernorm", [False, True], ids=["out_proj", "norm1+in_proj"])
def test_linear_backward_long_chain(lib, sms, layernorm, mode, with_tau):
    """fz_linear_backward at (2, 32, 128^3): out_proj (dy >= 0.1, m >= 0) and norm1 + in_proj (per-channel offsets on the
    input), against fp64 chunk by chunk; the bounds S as in test_mlp_backward_beyond_cap.  On the tensor cores this is a
    long chain below linear_bwd_tc2's 128-tile cap: 2 x 148 CTAs with 111 tiles (1776 MMAs) each on 148 SMs."""
    B, C, vox, eps = 2, 32, 128 ** 3, 1e-5
    tiles = B * (-(-vox // 128))
    nblk = min(tiles, 2 * sms)
    assert nblk * 128 >= tiles and -(-tiles // nblk) > 64, "linear_bwd_tc2: a long chain below its 128-tile cap"
    p = _glue_operands(B, C, 64, vox, 43)
    dev = p["x1"].device
    a = p["x1"] if layernorm else p["m"]
    resid = p["m"] if layernorm else None
    dy = p["dout"]
    da = torch.empty(B, C, vox, device=dev)
    dW, db, dg, dbt = (torch.empty(*s, device=dev) for s in ((C, C), (C,), (C,), (C,)))
    with _Glue(lib, mode):
        _check(lib.fz_linear_backward(_p(dy), _p(a), _p(p["g"]) if layernorm else None, _p(p["b"]) if layernorm else None,
                                      _p(p["w"]), _p(resid), _p(da), _p(dW), None if layernorm else _p(db),
                                      _p(dg) if layernorm else None, _p(dbt) if layernorm else None, B, C, vox,
                                      eps if layernorm else 0.0, int(layernorm), _st()))
    gm, bt, w = p["g"].double(), p["b"].double(), p["w"].double()
    z = lambda *s: torch.zeros(*s, device=dev, dtype=torch.float64)
    Q, SQ, sdy, Ssdy = z(C, C), z(C, C), z(C), z(C)
    da_ratio = 0.0
    for b, v in _chunks(B, vox):
        d, av = dy[b, :, v].double(), a[b, :, v].double()
        if layernorm:
            xh, rstd = _ln64(av, eps)
            want = _ln_back64(gm[:, None] * (w.t() @ d), xh, rstd) + resid[b, :, v].double()
        else:
            xh, want = av, w.t() @ d
        Q += d @ xh.t()
        SQ += d.abs() @ xh.abs().t()
        sdy += d.sum(1)
        Ssdy += d.abs().sum(1)
        da_ratio = max(da_ratio, _tol_ratio(da[b, :, v], want, 1e-4, 2e-5))
        del d, av, xh, want
    tag = f"{'norm1+in_proj' if layernorm else 'out_proj'} {'tcgen05' if mode == 7 else 'fp32-pipe'}"
    if layernorm:
        _assert_grad(dW, Q * gm[None, :] + sdy[:, None] * bt[None, :], SQ * gm.abs()[None, :] + Ssdy[:, None] * bt.abs()[None, :],
                     f"dW_in {tag}", with_tau)
        _assert_grad(dg, (w * Q).sum(0), (w.abs() * SQ).sum(0), f"dgamma {tag}", with_tau)
        _assert_grad(dbt, (w * sdy[:, None]).sum(0), (w.abs() * Ssdy[:, None]).sum(0), f"dbeta {tag}", with_tau)
    else:
        _assert_grad(dW, Q, SQ, f"dW_out {tag}", with_tau)
        _assert_grad(db, sdy, Ssdy, f"db_out {tag}", with_tau)
    assert da_ratio <= 1.0, f"da: max err / tol = {da_ratio:.3g} (rtol 1e-4, atol 2e-5)"


# ---- 4. buffers at a 4-byte offset ------------------------------------------------------------------------------------
def _unaligned(*shape, fill=None):
    """a contiguous tensor whose data starts 4 bytes past a 16-byte boundary"""
    n = math.prod(shape)
    buf = torch.randn(n + 4, device="cuda:0")
    t = buf[1:n + 1].view(*shape)
    if fill is not None:
        t.fill_(fill)
    assert t.is_contiguous() and t.data_ptr() % 16 == 4
    return t


def test_unaligned_buffers_are_refused_by_the_c_entry_points(lib):
    """fz_linear_wgrad (dy, x), fz_space_depth2 (in, out) and fz_conv3d_stem_forward (x, y) move 16-byte words: a buffer
    off a 16-byte boundary is FZ_ERR_UNSUPPORTED, before anything is written."""
    dev = torch.device("cuda:0")
    B, cin, cout, vox = 1, 64, 64, 4096
    ok_dy, ok_x = torch.randn(B, cout, vox, device=dev), torch.randn(B, cin, vox, device=dev)
    for mode in (7, 5):
        for dy, x in ((_unaligned(B, cout, vox), ok_x), (ok_dy, _unaligned(B, cin, vox))):
            dW = torch.full((cout, cin), SENTINEL, device=dev)
            db = torch.full((cout,), SENTINEL, device=dev)
            with _Glue(lib, mode), pytest.raises(NotImplementedError, match="aligned"):
                _check(lib.fz_linear_wgrad(_p(dy), _p(x), _p(dW), _p(db), B, cout, cin, vox, _st()))
            assert bool((dW == SENTINEL).all()) and bool((db == SENTINEL).all())
    full, patches = (2, 3, 8, 8, 16), (2, 24, 4 * 4 * 8)
    for to_depth in (1, 0):
        src_shape, dst_shape = (full, patches) if to_depth else (patches, full)
        for src, dst in ((_unaligned(*src_shape), torch.full(dst_shape, SENTINEL, device=dev)),
                         (torch.randn(src_shape, device=dev), _unaligned(*dst_shape, fill=SENTINEL))):
            with pytest.raises(NotImplementedError, match="aligned"):
                _check(lib.fz_space_depth2(_p(src), _p(dst), 2, 3, 8, 8, 16, to_depth, _st()))
            assert bool((dst == SENTINEL).all())
    w, bias = torch.randn(32, 4, 3, 3, 3, device=dev), torch.randn(32, device=dev)
    for x, y in ((_unaligned(1, 4, 8, 8, 8), torch.full((1, 32, 8, 8, 8), SENTINEL, device=dev)),
                 (torch.randn(1, 4, 8, 8, 8, device=dev), _unaligned(1, 32, 8, 8, 8, fill=SENTINEL))):
        with pytest.raises(NotImplementedError, match="aligned"):
            _check(lib.fz_conv3d_stem_forward(_p(x), _p(w), _p(bias), _p(y), 1, 4, 32, 8, 8, 8, _st()))
        assert bool((y == SENTINEL).all())
    torch.cuda.synchronize()


def _module_case(kind):
    import factorizer_b200 as ft
    from factorizer_b200 import layers
    if kind == "Linear":
        return ft.Linear(64, 96), (1, 64, 16, 16, 16), lambda x, p: F.conv1d(x.flatten(2), p[0], p[1]).view(1, 96, 16, 16, 16)
    if kind == "Conv3d-k2s2":
        return layers.Conv3d(32, 64, kernel_size=2, stride=2), (2, 32, 32, 32, 32), lambda x, p: F.conv3d(x, p[0], p[1], stride=2)
    if kind == "ConvTranspose3d-k2s2":
        return (layers.ConvTranspose3d(64, 32, kernel_size=2, stride=2), (2, 64, 16, 16, 16),
                lambda x, p: F.conv_transpose3d(x, p[0], p[1], stride=2))
    if kind == "stem-3x3x3":
        return layers.Conv3d(4, 32, kernel_size=3, padding=1), (2, 4, 32, 32, 32), lambda x, p: F.conv3d(x, p[0], p[1], padding=1)
    raise KeyError(kind)


@pytest.mark.parametrize("where", ["input", "output-gradient"])
@pytest.mark.parametrize("kind", ["Linear", "Conv3d-k2s2", "ConvTranspose3d-k2s2", "stem-3x3x3"])
def test_unaligned_views_through_the_layers(kind, where, monkeypatch):
    """A contiguous view at a 4-byte offset as the input, or as the gradient arriving from above: the layers take the
    torch formulation where a kernel needs 16-byte alignment, and output and all gradients match fp64 torch as in the
    other layer tests (rtol 1e-4 / atol 1e-5, gradients scaled by max(1, max|ref|)).  The offset gradient is seen to
    reach the backward that dispatches on it (the weight gradient, or the depth-to-space permutation's adjoint)."""
    from factorizer_b200 import _ops
    seen = []
    wgrad, run = _ops._channel_map_wgrad, _ops.SpaceDepth2._run

    def wgrad_spy(gy, x, want_bias):
        seen.append(gy.data_ptr())
        return wgrad(gy, x, want_bias)

    def run_spy(x, *args):
        seen.append(x.data_ptr())
        return run(x, *args)

    monkeypatch.setattr(_ops, "_channel_map_wgrad", wgrad_spy)
    monkeypatch.setattr(_ops.SpaceDepth2, "_run", staticmethod(run_spy))
    torch.manual_seed(51)
    dev = torch.device("cuda:0")
    mod, shape, ref_fn = _module_case(kind)
    mod = mod.to(dev)
    x = _unaligned(*shape) if where == "input" else torch.randn(shape, device=dev)
    x.requires_grad_(True)
    params = [q for q in mod.parameters()]
    keep = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False          # the library convolutions the layers fall back to, in full fp32
    try:
        y = mod(x)
        gy = _unaligned(*y.shape) if where == "output-gradient" else torch.randn(y.shape, device=dev)
        grads = torch.autograd.grad(y, [x] + params, gy)
        with torch.no_grad():
            y_inf = mod(x)
    finally:
        torch.backends.cudnn.allow_tf32 = keep
    if where == "output-gradient":
        assert any(q % 16 for q in seen), "the offset gradient did not reach the backward unchanged"
    x64 = x.detach().double().requires_grad_(True)
    p64 = [q.detach().double().requires_grad_(True) for q in params]
    y64 = ref_fn(x64, p64)
    refs = torch.autograd.grad(y64, [x64] + p64, gy.double())
    assert y.shape == y64.shape
    assert _tol_ratio(y, y64, 1e-4, 1e-5) <= 1.0, "y"
    assert _tol_ratio(y_inf, y64, 1e-4, 1e-5) <= 1.0, "no_grad y"
    for i, (g, r) in enumerate(zip(grads, refs)):
        assert g.shape == r.shape
        scale = max(1.0, float(r.abs().max()))
        assert _tol_ratio(g / scale, r / scale, 1e-4, 1e-5) <= 1.0, f"grad {i}"
