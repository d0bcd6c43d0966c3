"""GPU parity tests proper: every call goes through the C ABI (ctypes) and is compared with the
committed golden vectors produced by the reference, and with the numpy oracle on the same inputs.
Tolerances: bit-exact for matricize / inverse; rtol 1e-4 / atol 1e-5 (fp32) for NMF outputs and
input gradients, as BASELINE.json's north_star states."""
import numpy as np
import pytest
import torch
from torch import nn

import cases
from conftest import assert_close, tol_ratio
from oracle import factorizer_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ft():
    import factorizer_b200
    return factorizer_b200


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _np(t):
    return t.detach().cpu().numpy()


@pytest.mark.parametrize("name", list(cases.SW_CASES))
def test_swmatricize_bit_exact(ft, dev, golden, name):
    c = cases.SW_CASES[name]
    g = golden["sw"]
    mod = getattr(ft, c["cls"])((None, *c["x_shape"][1:]), **c["kw"])
    x = torch.from_numpy(cases.make_array(name, c["x_shape"], "randn")).to(dev)
    y = mod(x)
    assert tuple(y.shape) == tuple(g[f"{name}/y_shape"])
    assert cases.digest(_np(y)) == str(g[f"{name}/y_digest"])
    w = torch.from_numpy(cases.make_array(name, tuple(y.shape), "randn", tag="w")).to(dev)
    z = mod.inverse_forward(w)
    assert cases.digest(_np(z)) == str(g[f"{name}/z_digest"])
    rt = mod.inverse_forward(y)
    assert cases.digest(_np(rt)) == str(g[f"{name}/rt_digest"])
    assert bool(g[f"{name}/roundtrip_equal"]) == bool(torch.equal(rt, x))   # README.md:49-51


@pytest.mark.parametrize("name", list(cases.SW_CASES))
def test_swmatricize_autograd(ft, dev, name):
    """forward/inverse adjoints against the oracle (gradients of <w, f(x)>)."""
    c = cases.SW_CASES[name]
    mod = getattr(ft, c["cls"])((None, *c["x_shape"][1:]), **c["kw"])
    x_np = cases.make_array(name, c["x_shape"], "randn")
    x = torch.from_numpy(x_np).to(dev).requires_grad_(True)
    y = mod(x)
    w_np = cases.make_array(name, tuple(y.shape), "randn", tag="w")
    w = torch.from_numpy(w_np).to(dev).requires_grad_(True)
    (gx,) = torch.autograd.grad((y * w).sum(), x)
    z = mod.inverse_forward(w)
    (gw,) = torch.autograd.grad((z * x.detach()).sum(), w)
    kw = dict(c["kw"])
    shifts = kw.pop("shifts", None)
    H, d, grid, patch = O.resolve_geometry((None, *c["x_shape"][1:]), **kw)
    n = len(c["x_shape"]) - 2
    if c["cls"] == "SWMatricize":
        shifts = O.normalise_shifts(O.default_shifts(patch) if shifts is None else shifts, n)
        S = len(shifts)
        parts = np.split(w_np, S, axis=0)
        gx_ref = sum(O.unmatricize(p, x_np.shape[0], H, d, grid, patch, s) for p, s in zip(parts, shifts))
        gw_ref = O.swmat_forward(x_np / np.float32(S), H, d, grid, patch, shifts)
    else:
        shifts = O.normalise_shifts([shifts], n)
        gx_ref = O.unmatricize(w_np, x_np.shape[0], H, d, grid, patch, shifts[0])
        gw_ref = O.swmat_forward(x_np, H, d, grid, patch, shifts)
    assert_close(_np(gx), gx_ref, rtol=1e-6, atol=1e-6, what="gx")
    np.testing.assert_array_equal(_np(gw), gw_ref)


WELL_CONDITIONED = {n for n, c in cases.NMF_CASES.items() if c["solver"] == "mu" or c["rank"] == 1}


@pytest.mark.parametrize("name", list(cases.NMF_CASES))
def test_nmf_matches_reference(ft, dev, golden, name):
    c = cases.NMF_CASES[name]
    g = golden["nmf"]
    M, N = c["shape"][-2:]
    nmf = ft.NMF(size=(M, N), rank=c["rank"], num_iters=c["num_iters"], num_grad_steps=c["num_grad_steps"],
                 init="uniform", solver=c["solver"])
    nmf.load_state_dict({"init.u0": torch.from_numpy(g[f"{name}/u0"]), "init.v0": torch.from_numpy(g[f"{name}/v0"])})
    nmf = nmf.to(dev)
    x = torch.from_numpy(cases.make_array(name, c["shape"], c["dist"])).to(dev).requires_grad_(True)
    gy = torch.from_numpy(cases.make_array(name, c["shape"], "randn", tag="gy")).to(dev)
    y = nmf(x)                                               # fused decompose + reconstruct
    (gx,) = torch.autograd.grad((y * gy).sum(), x)
    u, v = nmf.decompose(x)                                  # factor outputs + their own backward
    y2 = nmf.reconstruct(u, v)
    (gx2,) = torch.autograd.grad((y2 * gy).sum(), x)
    assert u.shape == (*c["shape"][:-2], M, c["rank"]) and v.shape == (*c["shape"][:-2], N, c["rank"])
    assert (u >= 0).all() and (v >= 0).all()                 # reference tests/test_nmf.py:19-20
    assert y.shape == x.shape
    if name in WELL_CONDITIONED:
        assert_close(_np(u), g[f"{name}/u"], what="u")
        assert_close(_np(v), g[f"{name}/v"], what="v")
        assert_close(_np(y), g[f"{name}/y"], what="y")
        assert_close(_np(y2), g[f"{name}/y"], what="y via decompose")
        assert_close(_np(gx), g[f"{name}/gx"], what="gx")
        assert_close(_np(gx2), g[f"{name}/gx"], what="gx via decompose")
    else:
        ref_gap = max(tol_ratio(g[f"{name}/y"], g[f"{name}/y64"]), tol_ratio(g[f"{name}/gx"], g[f"{name}/gx64"]))
        for yy, gg in ((y, gx), (y2, gx2)):
            ours = max(tol_ratio(_np(yy), g[f"{name}/y64"]), tol_ratio(_np(gg), g[f"{name}/gx64"]))
            assert ours <= max(1.0, 10 * ref_gap), (ours, ref_gap)


def _fused_module(ft, c, g, name, dev):
    xs = c["x_shape"]
    reshape = getattr(ft, c["cls"])((None, *xs[1:]), **c["kw"])
    nmf = ft.NMF(reshape.output_size[2:], init="uniform", **c["nmf"])
    nmf.load_state_dict({"init.u0": torch.from_numpy(g[f"{name}/u0"]), "init.v0": torch.from_numpy(g[f"{name}/v0"])})
    return reshape, nmf.to(dev)


@pytest.mark.parametrize("path", ["auto", "pipeline", "three-launch", "window", "generic"])
@pytest.mark.parametrize("name", list(cases.FUSED_CASES))
def test_fused_core_matches_reference(ft, dev, golden, name, path):
    """Every kernel family that covers a case, selected per call through fz_geom.path: the automatic choice, the octant
    kernels as one pipelined launch and as three launches, the window-at-a-time / sub-warp kernels, the generic ones."""
    from factorizer_b200 import _lib, _ops
    c = cases.FUSED_CASES[name]
    g = golden["fused"]
    reshape, nmf = _fused_module(ft, c, g, name, dev)
    x = torch.from_numpy(cases.make_array(name, c["x_shape"], c["dist"])).to(dev).requires_grad_(True)
    gy = torch.from_numpy(cases.make_array(name, c["x_shape"], "randn", tag="gy")).to(dev)
    reshape._geom.path = {"auto": _lib.FZ_PATH_AUTO, "pipeline": _lib.FZ_PATH_OCTANT_PIPELINE, "three-launch": _lib.FZ_PATH_OCTANT_3LAUNCH,
                          "window": _lib.FZ_PATH_NO_OCTANT, "generic": _lib.FZ_PATH_GENERIC}[path]
    y = _ops.SWNMF.apply(x, nmf.init.u0, nmf.init.v0, reshape._geom, nmf.solver_spec(), c["relu"])
    took = _lib.lib().fz_last_path()
    (gx,) = torch.autograd.grad((y * gy).sum(), x)
    if path == "pipeline" and name in ("fused_cfg2_16", "fused_cfg2_24_b2", "fused_k2"):
        assert took == 6
    if path == "three-launch" and name in ("fused_cfg2_16", "fused_cfg2_24_b2", "fused_k2"):
        assert took == 2
    assert_close(_np(y), g[f"{name}/y"], what="y")
    assert_close(_np(gx), g[f"{name}/gx"], what="gx")


def test_kernel_path_selection(ft, dev, golden):
    """Which kernel family serves which geometry (fz_last_path): 2 = three-pass octant kernels (default Swin
    geometry), 4 = the same per pair of window sets on a rolled volume (brats23 shifts), 1 = window-at-a-time 8x512
    kernels (any other shifts), 3 = sub-warp register kernels (64-column
    windows of the isles22 bundle / reference tests, small ft.NMF batches), 5 = one grid-wide pass per sweep for the
    huge matrices of Matricize(grid_size=1), 0 = generic shared-memory kernels."""
    from factorizer_b200 import _lib, _ops
    lib = _lib.lib()
    want = {"fused_cfg2_16": 2, "fused_brats_s4": 4, "fused_isles_s4": 3, "fused_nh8_ps4": 3, "fused_2d": 3,
            "fused_mu_r2": 0, "fused_global_mu": 0, "fused_global_mu_big": 5, "fused_global_hals_big": 5,
            "fused_global_mu_k2": 5}
    for name, path in want.items():
        c = cases.FUSED_CASES[name]
        reshape, nmf = _fused_module(ft, c, golden["fused"], name, dev)
        x = torch.from_numpy(cases.make_array(name, c["x_shape"], c["dist"])).to(dev)
        _ops.SWNMF.apply(x, nmf.init.u0, nmf.init.v0, reshape._geom, nmf.solver_spec(), c["relu"])
        assert lib.fz_last_path() == path, (name, lib.fz_last_path())
    nmf = ft.NMF(size=(16, 64), rank=1, solver="mu").to(dev)
    nmf(torch.rand(3, 16, 64, device=dev))
    assert lib.fz_last_path() == 3


@pytest.mark.parametrize("name", ["fused_cfg2_16", "fused_mu_r2"])
def test_unfused_chain_equals_fused(ft, dev, golden, name):
    """reshape -> act -> factorize -> inverse through the standalone kernels agrees with the fused op."""
    from factorizer_b200 import _ops
    c = cases.FUSED_CASES[name]
    g = golden["fused"]
    reshape, nmf = _fused_module(ft, c, g, name, dev)
    x = torch.from_numpy(cases.make_array(name, c["x_shape"], c["dist"])).to(dev).requires_grad_(True)
    gy = torch.from_numpy(cases.make_array(name, c["x_shape"], "randn", tag="gy")).to(dev)
    m = reshape(x)
    if c["relu"]:
        m = torch.relu(m)
    y = reshape.inverse_forward(nmf(m))
    (gx,) = torch.autograd.grad((y * gy).sum(), x)
    assert_close(_np(y), g[f"{name}/y"], what="y")
    assert_close(_np(gx), g[f"{name}/gx"], what="gx")


@pytest.mark.parametrize("name", list(cases.BLOCK_CASES))
def test_factorizer_block_matches_reference(ft, dev, golden, name):
    c = cases.BLOCK_CASES[name]
    g = golden["block"]
    # shapes the channel-map kernel does not take fall back to library GEMMs, which may default to TF32 on CUDA;
    # parity against the reference's fp32 CPU run needs true fp32 there (our own kernels never use one TF32 pass)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    blk = ft.FactorizerBlock(channels=c["channels"], spatial_size=c["spatial"], norm=ft.LayerNorm,
                             reshape=(ft.SWMatricize, c["kw"]), act=nn.ReLU, factorize=ft.NMF,
                             mlp_ratio=c["mlp_ratio"], dropout=0.0, **c["nmf"])
    sd = {k.split("/sd/")[1]: torch.from_numpy(g[k]) for k in g if k.startswith(name + "/sd/")}
    blk.load_state_dict(sd)
    blk = blk.to(dev)
    xs = (c["batch"], c["channels"], *c["spatial"])
    x = torch.from_numpy(cases.make_array(name, xs, "randn")).to(dev).requires_grad_(True)
    gy = torch.from_numpy(cases.make_array(name, xs, "randn", tag="gy")).to(dev)
    assert blk._fused_args(x) is not None
    y = blk(x)
    assert type(y.grad_fn).__name__ == ("FactorizerBlockFnBackward" if c["channels"] == 32 else "FactorizerBlockWideFnBackward")
    params = dict(blk.named_parameters())
    grads = torch.autograd.grad((y * gy).sum(), [x] + list(params.values()))
    assert_close(_np(y), g[f"{name}/y"], what="y")
    assert_close(_np(grads[0]), g[f"{name}/gx"], what="gx")
    for (k, _), gp in zip(params.items(), grads[1:]):
        ref = g[f"{name}/gp/{k}"]
        # parameter gradients are sums over thousands of voxels of fp32 products: scale the bound accordingly
        scale = max(1.0, float(np.abs(ref).max()))
        assert_close(_np(gp) / scale, ref / scale, rtol=1e-4, atol=1e-4, what=f"grad {k}")
    # inference path (no saved tensors) gives the same output
    with torch.no_grad():
        assert torch.equal(blk(x.detach()), y.detach())


@pytest.mark.parametrize("name", list(cases.MODEL_CASES))
def test_factorizer_model_matches_reference(ft, dev, golden, name):
    """Whole Swin Factorizer (BASELINE config 4/5 architecture at a small size) from a reference state_dict:
    output, input gradient and every parameter gradient against the reference's CPU run."""
    c, g = cases.MODEL_CASES[name], golden["model"]
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    net = ft.Factorizer(in_channels=c["in_channels"], out_channels=c["out_channels"], spatial_size=c["spatial"],
                        norm=ft.LayerNorm, reshape=(ft.SWMatricize, c["reshape_kw"]), act=nn.ReLU, factorize=ft.NMF,
                        **c["kw"])
    net.load_state_dict({k.split("/sd/")[1]: torch.from_numpy(g[k]) for k in g if k.startswith(name + "/sd/")})
    net = net.to(dev).eval()
    xs = (c["batch"], c["in_channels"], *c["spatial"])
    x = torch.from_numpy(cases.make_array(name, xs, "randn")).to(dev).requires_grad_(True)
    y = net(x)
    assert tuple(y.shape) == g[f"{name}/y"].shape
    gy = torch.from_numpy(cases.make_array(name, tuple(y.shape), "randn", tag="gy")).to(dev)
    params = dict(net.named_parameters())
    grads = torch.autograd.grad((y * gy).sum(), [x] + list(params.values()))
    assert_close(_np(y), g[f"{name}/y"], what="y")
    assert_close(_np(grads[0]), g[f"{name}/gx"], what="gx")
    for (k, _), gp in zip(params.items(), grads[1:]):
        ref = g[f"{name}/gp/{k}"]
        scale = max(1.0, float(np.abs(ref).max()))
        assert_close(_np(gp) / scale, ref / scale, rtol=2e-4, atol=2e-4, what=f"grad {k}")


def test_block_path_choice_and_edge_inputs(ft, dev):
    """README.md:56-73 block (dropout 0.1): training mode keeps the layer-by-layer path (dropout masks come from
    torch), eval mode and dropout 0 take the fused kernels and agree with the layer-by-layer result; an empty batch
    and a non-contiguous input go through the fused path too."""
    torch.manual_seed(5)
    mk = lambda p: ft.FactorizerBlock(channels=32, spatial_size=(8, 8, 16), norm=ft.LayerNorm,
                                      reshape=(ft.SWMatricize, {"head_dim": 8, "patch_size": 8}), act=nn.ReLU,
                                      factorize=ft.NMF, rank=1, num_iters=5, init="uniform", solver="hals", mlp_ratio=2,
                                      dropout=p).to(dev)
    blk = mk(0.1)
    x = torch.randn(2, 32, 8, 8, 16, device=dev, requires_grad=True)
    assert blk.training and blk._fused_args(x) is None
    assert torch.isfinite(blk(x)).all()
    blk.eval()
    assert blk._fused_args(x) is not None
    y = blk(x)
    (gx,) = torch.autograd.grad(y.square().sum(), x)
    # the same block, layer by layer (fused core + library GEMMs), as the reference composes it
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    y2 = x + blk.fact(blk.norm1(x))
    y2 = y2 + blk.mlp(blk.norm2(y2))
    (gx2,) = torch.autograd.grad(y2.square().sum(), x)
    assert_close(_np(y), _np(y2), what="fused vs layer-by-layer y")
    assert_close(_np(gx), _np(gx2), rtol=2e-4, atol=2e-4, what="fused vs layer-by-layer gx")
    # non-contiguous input view
    xt = torch.randn(2, 32, 8, 16, 8, device=dev).transpose(3, 4)
    assert not xt.is_contiguous()
    assert torch.equal(blk(xt), blk(xt.contiguous()))
    # empty batch
    e = blk(torch.empty(0, 32, 8, 8, 16, device=dev))
    assert e.shape == (0, 32, 8, 8, 16)


def _glue_call(fn, *args):
    from factorizer_b200 import _lib as L
    L.check(fn(*[a.data_ptr() if isinstance(a, torch.Tensor) else a for a in args]))


@pytest.fixture(params=[0, 5, 7], ids=["fp32-pipe", "tc-mlp", "tc-mlp+linear-wgrad"])
def glue_mode(request):
    """0 = every glue kernel on the FP32 pipe; bit 0 = forward MLP kernel on tcgen05, bit 2 = MLP backward on tcgen05, bit 1 =
    also linear_bwd's weight gradient and fz_linear_wgrad (7, all three, is the default)."""
    from factorizer_b200 import _lib as L
    lib = L.lib()
    before = lib.fz_get_glue_mode()
    lib.fz_set_glue_mode(request.param)
    yield request.param
    lib.fz_set_glue_mode(before)


@pytest.mark.parametrize("HID", [32, 48, 64, 128, 136, 256])
@pytest.mark.parametrize("shape", [(1, 32, 8, 8, 8), (2, 32, 6, 10, 7), (3, 32, 1030), (2, 32, 30002)])
def test_glue_kernels_against_torch_fp64(ft, dev, shape, HID, glue_mode):
    """Each kernel of csrc/fz_block_glue*.cu through the C ABI against fp64 torch autograd of the same
    layers (LayerNorm over channels, k=1 Conv1d, exact GELU: the reference's factorizer/layers/*).  The last shape gives
    every persistent CTA several tiles (470 tiles of 128 voxels on 148 SMs)."""
    from factorizer_b200 import _lib as L
    lib = L.lib()
    torch.manual_seed(3)
    B, C = shape[0], shape[1]
    vox = int(np.prod(shape[2:]))
    if vox % 2:
        pytest.skip("odd voxel count")
    st = torch.cuda.current_stream().cuda_stream
    r = lambda *s: torch.randn(*s, device=dev)
    x, m, gout = 2 * r(B, C, vox) + 0.5, r(B, C, vox), r(B, C, vox)
    g1, b1n, g2, b2n = 1 + 0.3 * r(C), 0.3 * r(C), 1 + 0.3 * r(C), 0.3 * r(C)
    w_in, w_out, b_out = r(C, C) / 6, r(C, C) / 6, 0.2 * r(C)
    w1, bb1, w2, bb2 = r(HID, C) / 6, 0.2 * r(HID), r(C, HID) / 7, 0.2 * r(C)
    eps = 1e-5
    D = lambda t: t.detach().double().requires_grad_(True)
    F = torch.nn.functional
    ln = lambda t, g, b: F.layer_norm(t.movedim(1, -1), (C,), g, b, eps).movedim(-1, 1)
    lin = lambda t, w, b=None: torch.einsum("oc,bcv->bov", w, t) + (0 if b is None else b[None, :, None])

    def close(a, b, what, scale=1.0):
        assert_close(_np(a) / scale, _np(b) / scale, rtol=1e-4, atol=2e-5, what=what)

    # ---- z = W_in LN1(x) and its backward (with a residual gradient) ----
    z = torch.empty_like(x)
    _glue_call(lib.fz_ln_linear_forward, x, g1, b1n, w_in, z, B, C, vox, eps, st)
    xd, g1d, b1d, wind = D(x), D(g1), D(b1n), D(w_in)
    zd = lin(ln(xd, g1d, b1d), wind)
    close(z, zd, "z")
    dz, resid = r(B, C, vox), r(B, C, vox)
    ref = torch.autograd.grad((zd * dz.double()).sum() + (xd * resid.double()).sum(), [xd, wind, g1d, b1d])
    dx, dw, dg, dbt = torch.empty_like(x), torch.empty_like(w_in), torch.empty_like(g1), torch.empty_like(b1n)
    _glue_call(lib.fz_linear_backward, dz, x, g1, b1n, w_in, resid, dx, dw, None, dg, dbt, B, C, vox, eps, 1, st)
    close(dx, ref[0], "dx (in_proj + norm1)")
    for got, want, what in ((dw, ref[1], "dW_in"), (dg, ref[2], "dgamma1"), (dbt, ref[3], "dbeta1")):
        close(got, want, what, scale=max(1.0, float(want.abs().max())))

    # ---- out_proj backward (no LayerNorm, bias) ----
    md, woutd, boutd = D(m), D(w_out), D(b_out)
    yd = lin(md, woutd, boutd)
    ref = torch.autograd.grad((yd * dz.double()).sum(), [md, woutd, boutd])
    dm, dwo, dbo = torch.empty_like(x), torch.empty_like(w_out), torch.empty_like(b_out)
    _glue_call(lib.fz_linear_backward, dz, m, None, None, w_out, None, dm, dwo, dbo, None, None, B, C, vox, 0.0, 0, st)
    close(dm, ref[0], "dm")
    for got, want, what in ((dwo, ref[1], "dW_out"), (dbo, ref[2], "db_out")):
        close(got, want, what, scale=max(1.0, float(want.abs().max())))

    # ---- x1 = x + out_proj(m); out = x1 + MLP(LN2(x1)) and the MLP backward ----
    x1, out = torch.empty_like(x), torch.empty_like(x)
    _glue_call(lib.fz_mixer_mlp_forward, x, m, w_out, b_out, g2, b2n, w1, bb1, w2, bb2, x1, out, B, C, HID, vox, eps, st)
    x1d = (x.double() + lin(m.double(), w_out.double(), b_out.double())).detach().requires_grad_(True)
    g2d, b2d, w1d, bb1d, w2d, bb2d = D(g2), D(b2n), D(w1), D(bb1), D(w2), D(bb2)
    outd = x1d + lin(F.gelu(lin(ln(x1d, g2d, b2d), w1d, bb1d)), w2d, bb2d)
    close(x1, x1d, "x1")
    close(out, outd, "out")
    out2 = torch.empty_like(x)
    _glue_call(lib.fz_mixer_mlp_forward, x, m, w_out, b_out, g2, b2n, w1, bb1, w2, bb2, None, out2, B, C, HID, vox, eps, st)
    assert torch.equal(out, out2)
    ref = torch.autograd.grad((outd * gout.double()).sum(), [x1d, g2d, b2d, w1d, bb1d, w2d, bb2d])
    dx1 = torch.empty_like(x)
    got = [dx1] + [torch.empty_like(t) for t in (g2, b2n, w1, bb1, w2, bb2)]
    _glue_call(lib.fz_mlp_backward, x1, gout, g2, b2n, w1, bb1, w2, *got, B, C, HID, vox, eps, st)
    close(got[0], ref[0], "dx1")
    for a, b, what in zip(got[1:], ref[1:], ("dgamma2", "dbeta2", "dW1", "db1", "dW2", "db2")):
        close(a, b, what, scale=max(1.0, float(b.abs().max())))


def test_glue_rejects_unsupported(ft, dev):
    from factorizer_b200 import _lib as L
    lib = L.lib()
    assert lib.fz_glue_supported(32, 64, 512) == 1
    assert lib.fz_glue_supported(16, 32, 512) == 0 and lib.fz_glue_supported(32, 128, 512) == 1
    assert lib.fz_glue_supported(32, 264, 512) == 0 and lib.fz_glue_supported(32, 60, 512) == 0
    assert lib.fz_glue_supported(32, 64, 511) == 0
    x = torch.zeros(1, 16, 64, device=dev)
    with pytest.raises(NotImplementedError):
        L.check(lib.fz_ln_linear_forward(x.data_ptr(), None, None, x.data_ptr(), x.data_ptr(), 1, 16, 64, 1e-5, None))


def test_reference_test_nmf_port(ft, dev):
    """Port of the reference's tests/test_nmf.py:7-39 onto CUDA tensors."""
    size = (2, 4, 8, 16)
    nmf = ft.NMF(size=(8, 16), rank=3, init="uniform", solver="hals").to(dev)
    x = torch.rand(size, device=dev, requires_grad=True)
    u, v = nmf.decompose(x)
    assert u.shape == (2, 4, 8, 3) and v.shape == (2, 4, 16, 3)
    assert (u >= 0).all() and (v >= 0).all()
    assert nmf(x).shape == x.shape
    u = torch.rand((2, 4, 8, 3), device=dev, requires_grad=True)
    v = torch.rand((2, 4, 16, 3), device=dev, requires_grad=True)
    assert nmf.reconstruct(u, v).shape == size
    loss = nmf.loss(x, u, v)
    assert loss.shape == size[:1] and (loss >= 0).all()


def test_standalone_nmf_on_large_matrices(ft, dev, golden):
    """ft.NMF on matrices beyond a CTA's shared memory (rank 1): forward and input gradient against the reference
    golden of the identical computation through Matricize(num_heads=1, grid_size=1), which is a pure view."""
    from factorizer_b200 import _lib
    name = "fused_global_mu_big"
    c = cases.FUSED_CASES[name]
    gold = golden["fused"]
    xs = c["x_shape"]
    M, N = xs[1], int(np.prod(xs[2:]))
    nmf = ft.NMF(size=(M, N), rank=1, num_iters=5, init="uniform", solver="mu")
    nmf.load_state_dict({"init.u0": torch.from_numpy(gold[f"{name}/u0"]), "init.v0": torch.from_numpy(gold[f"{name}/v0"])})
    nmf = nmf.to(dev)
    x = torch.from_numpy(cases.make_array(name, xs, c["dist"])).to(dev).reshape(xs[0], M, N).requires_grad_(True)
    gy = torch.from_numpy(cases.make_array(name, xs, "randn", tag="gy")).to(dev).reshape(xs[0], M, N)
    y = nmf(x)                       # x >= 0 here, so the golden's ReLU is the identity
    assert _lib.lib().fz_last_path() == 5
    (gx,) = torch.autograd.grad((y * gy).sum(), x)
    assert_close(_np(y).reshape(xs), gold[f"{name}/y"], what="y")
    assert_close(_np(gx).reshape(xs), gold[f"{name}/gx"], what="gx")


def test_empty_batch(ft, dev):
    nmf = ft.NMF(size=(8, 16), rank=1).to(dev)
    y = nmf(torch.empty(0, 8, 16, device=dev))
    assert y.shape == (0, 8, 16)


def test_full_size_properties(ft, dev):
    """BASELINE config 2 at its real size (1,32,128^3): size-independent properties.
    (a) exact round trip of SWMatricize (README.md:49-51); (b) every window is independent and the
    same u0/v0 serve all of them, so a volume tiled from one 8^3 window pattern per head gives an
    output that is the same tiling; (c) HALS rank-1 of a rank-1 non-negative window reproduces it."""
    from factorizer_b200 import _ops
    C, n = 32, 128
    sw = ft.SWMatricize((None, C, n, n, n), head_dim=8, patch_size=8)
    torch.manual_seed(0)
    x = torch.rand(1, C, n, n, n, device=dev)
    y = sw(x)
    assert y.shape == (8, 4096, 8, 512)
    assert torch.equal(sw.inverse_forward(y), x)
    del y
    nmf = ft.NMF((8, 512), rank=1, num_iters=5, init="uniform", solver="hals").to(dev)
    # (b) periodic volume with period 8 along every axis: shifted and unshifted windows all see a
    # cyclic shift of the same matrix set, outputs must be periodic too
    tile = torch.rand(1, C, 8, 8, 8, device=dev)
    xp = tile.repeat(1, 1, 16, 16, 16).contiguous()
    yp = _ops.SWNMF.apply(xp, nmf.init.u0, nmf.init.v0, sw._geom, nmf.solver_spec(), True)
    ref = yp[:, :, :8, :8, :8].repeat(1, 1, 16, 16, 16)
    assert torch.allclose(yp, ref, rtol=1e-5, atol=1e-6)
    small = ft.SWMatricize((None, C, 8, 8, 8), head_dim=8, patch_size=8)
    ys = _ops.SWNMF.apply(tile.contiguous(), nmf.init.u0, nmf.init.v0, small._geom, nmf.solver_spec(), True)
    assert torch.allclose(yp[:, :, :8, :8, :8], ys, rtol=1e-4, atol=1e-5)
    # (c) rank-1 windows are fixed points: a (channel) x b (voxel) with constant b over space
    a = torch.rand(1, C, 1, 1, 1, device=dev) + 0.5
    x1 = a.expand(1, C, n, n, n).contiguous()
    y1 = _ops.SWNMF.apply(x1, nmf.init.u0, nmf.init.v0, sw._geom, nmf.solver_spec(), True)
    assert torch.allclose(y1, x1, rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("shape", [(2, 32, 8, 8, 8), (1, 16, 6, 10, 4), (3, 8, 50), (1, 32, 16, 16, 16),
                                   (2, 64, 16, 16, 16), (1, 24, 6, 10, 4), (2, 128, 8, 8, 8), (3, 512, 4, 4, 4), (1, 5, 7, 6),
                                   (1, 256, 2, 33, 1), (1, 200, 6, 6, 6), (2, 72, 10, 10, 2), (1, 64, 64, 64, 32)])
def test_layernorm_channels_first(ft, dev, shape):
    """ft.LayerNorm (hand-written channels-first kernel) against torch's own layer_norm on the permuted
    tensor, which is literally what the reference does (factorizer/layers/norm.py:25-34): output, input
    gradient and the affine parameters' gradients."""
    from factorizer_b200 import _ops
    torch.manual_seed(0)
    C = shape[1]
    ln = ft.LayerNorm(C).to(dev)
    with torch.no_grad():
        ln.norm.weight.copy_(torch.randn(C, device=dev))
        ln.norm.bias.copy_(torch.randn(C, device=dev))
    x = (3 * torch.randn(shape, device=dev) + 1).requires_grad_(True)
    gy = torch.randn(shape, device=dev)
    assert _ops.layernorm_cf_supported(x)
    y = ln(x)
    gx, gw, gb = torch.autograd.grad((y * gy).sum(), [x, ln.norm.weight, ln.norm.bias])
    x64 = x.detach().double().requires_grad_(True)
    w64 = ln.norm.weight.detach().double().requires_grad_(True)
    b64 = ln.norm.bias.detach().double().requires_grad_(True)
    y64 = torch.nn.functional.layer_norm(x64.movedim(1, -1), (C,), w64, b64, ln.norm.eps).movedim(-1, 1)
    rx, rw, rb = torch.autograd.grad((y64 * gy.double()).sum(), [x64, w64, b64])
    assert_close(_np(y), _np(y64), what="y")
    assert_close(_np(gx), _np(rx), what="gx")
    scale = max(1.0, float(rw.abs().max()), float(rb.abs().max()))
    assert_close(_np(gw) / scale, _np(rw) / scale, what="gw")
    assert_close(_np(gb) / scale, _np(rb) / scale, what="gb")


@pytest.mark.parametrize("shape", [(2, 32, 8, 8, 8), (1, 64, 6, 10, 4), (3, 200, 50), (1, 512, 8, 8, 8), (2, 8, 4098)])
def test_layernorm_backward_with_residual_gradient(ft, dev, shape):
    """fz_layernorm_cf_backward_add: dx = add + LN'(dy) in one pass (every kernel family: register kernels for 8 / 16 / 32
    channels, the chunked one, the sliced one for few voxels) against torch fp64; d(gamma), d(beta) as without the addend."""
    from factorizer_b200 import _lib as L
    lib = L.lib()
    torch.manual_seed(21)
    B, C = shape[0], shape[1]
    x = torch.randn(shape, device=dev)
    vox = x.numel() // (B * C)
    gamma, beta = torch.randn(C, device=dev), torch.randn(C, device=dev)
    gy, add = torch.randn(shape, device=dev), torch.randn(shape, device=dev)
    dx, dg, db = torch.full_like(x, float("nan")), torch.empty(C, device=dev), torch.empty(C, device=dev)
    L.check(lib.fz_layernorm_cf_backward_add(x.data_ptr(), gamma.data_ptr(), gy.data_ptr(), add.data_ptr(), dx.data_ptr(), dg.data_ptr(),
                                             db.data_ptr(), B, C, vox, 1e-5, torch.cuda.current_stream().cuda_stream))
    x64 = x.double().requires_grad_(True)
    g64, b64 = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    y64 = torch.nn.functional.layer_norm(x64.movedim(1, -1), (C,), g64, b64, 1e-5).movedim(-1, 1)
    rx, rg, rb = torch.autograd.grad((y64 * gy.double()).sum(), [x64, g64, b64])
    assert_close(_np(dx), _np(rx + add.double()), what="dx")
    scale = max(1.0, float(rg.abs().max()), float(rb.abs().max()))
    assert_close(_np(dg) / scale, _np(rg) / scale, what="d gamma")
    assert_close(_np(db) / scale, _np(rb) / scale, what="d beta")


@pytest.mark.parametrize("shape,cout,bias", [((1, 64, 32, 32, 32), 128, True), ((2, 96, 8200), 64, True),
                                             ((1, 32, 40, 40, 12), 32, False), ((3, 128, 24, 24, 24), 256, True),
                                             ((1, 96, 32, 32, 32), 40, True), ((2, 200, 32, 32, 16), 32, True)])
def test_linear_weight_gradient_kernel(ft, dev, shape, cout, bias):
    """ft.Linear on long voxel axes: output and input gradient are library GEMMs, the weight / bias gradients come
    from csrc/fz_linear.cu; all four against the reference's formulation (a k=1 Conv1d, layers/linear.py:53-58) in
    fp64."""
    from factorizer_b200 import _ops
    torch.manual_seed(3)
    lin = ft.Linear(shape[1], cout, bias=bias).to(dev)
    x = torch.randn(shape, device=dev, requires_grad=True)
    gy = torch.randn(shape[0], cout, *shape[2:], device=dev)
    assert _ops.linear_wgrad_supported(x.flatten(2), cout)
    y = lin(x)
    params = [lin.linear.weight] + ([lin.linear.bias] if bias else [])
    grads = torch.autograd.grad((y * gy).sum(), [x] + params)
    x64 = x.detach().double().requires_grad_(True)
    p64 = [p.detach().double().requires_grad_(True) for p in params]
    y64 = torch.nn.functional.conv1d(x64.flatten(2), p64[0], p64[1] if bias else None).view(gy.shape)
    refs = torch.autograd.grad((y64 * gy.double()).sum(), [x64] + p64)
    assert_close(_np(y), _np(y64), what="y")
    for name, g, r in zip(["gx", "gw", "gb"], grads, refs):
        assert g.shape == r.shape
        scale = max(1.0, float(r.abs().max()))
        assert_close(_np(g) / scale, _np(r) / scale, what=name)
    # short voxel axes and odd channel counts stay with the library path
    assert not _ops.linear_wgrad_supported(torch.randn(1, 64, 8, 8, 8, device=dev).flatten(2), 64)
    assert not _ops.linear_wgrad_supported(torch.randn(1, 48, 31, 31, 31, device=dev).flatten(2), 40)


@pytest.mark.parametrize("B,cin,cout,vox,bias", [(1, 64, 64, 4096, True), (2, 96, 40, 8200, True), (1, 512, 512, 516, False),
                                                 (3, 40, 200, 1028, True), (1, 32, 3, 32768, True), (2, 256, 128, 4100, False),
                                                 (1, 4, 16, 64, True), (1, 136, 72, 260, True)])
def test_channel_map_tensor_core_kernel(ft, dev, B, cin, cout, vox, bias):
    """fz_linear_forward (csrc/fz_linear_tc.cu: tcgen05, 3xTF32, segmented accumulation) through the C ABI against the
    reference's formulation (a k=1 Conv1d, layers/linear.py:53-58) in fp64: ragged voxel tiles, channel counts that are not
    multiples of the K chunk / output tile, several samples, long K (512 channels = 48 accumulation steps per accumulator)."""
    from factorizer_b200 import _lib as L
    lib = L.lib()
    torch.manual_seed(11)
    x = torch.randn(B, cin, vox, device=dev)
    W = torch.randn(cout, cin, device=dev) / cin ** 0.5
    b = torch.randn(cout, device=dev) if bias else None
    y = torch.full((B, cout, vox), float("nan"), device=dev)
    assert lib.fz_linear_forward_supported(cout, cin, vox)
    L.check(lib.fz_linear_forward(x.data_ptr(), W.data_ptr(), b.data_ptr() if bias else None, y.data_ptr(), B, cin, cout, vox,
                                  torch.cuda.current_stream().cuda_stream))
    ref = torch.nn.functional.conv1d(x.double(), W.double().unsqueeze(-1), b.double() if bias else None)
    assert_close(_np(y), _np(ref), what="y")
    # fused epilogues (fz_linear_forward_ex): + residual | r and gelu(r) | r * gelu'(aux)
    aux = torch.randn(B, cout, vox, device=dev)
    y2 = torch.full_like(y, float("nan"))
    st = torch.cuda.current_stream().cuda_stream
    run = lambda epi: L.check(lib.fz_linear_forward_ex(x.data_ptr(), W.data_ptr(), b.data_ptr() if bias else None, y.data_ptr(), B, cin,
                                                       cout, vox, epi, 0, aux.data_ptr(), y2.data_ptr(), st))
    run(1)
    assert_close(_np(y), _np(ref + aux.double()), what="residual epilogue")
    run(2)
    assert_close(_np(y), _np(ref), what="GELU epilogue, pre-activation")
    assert_close(_np(y2), _np(torch.nn.functional.gelu(ref)), what="GELU epilogue, activation")
    run(4)
    assert_close(_np(y), _np(torch.nn.functional.gelu(ref)), what="GELU-only epilogue")
    run(3)
    a64 = aux.double().requires_grad_(True)
    (gp,) = torch.autograd.grad(torch.nn.functional.gelu(a64).sum(), a64)
    assert_close(_np(y), _np(ref * gp), what="GELU-gradient epilogue")
    # the weight read transposed (the input gradient from the layer's weight as stored): Wt is (cin, cout) row-major
    if cout % 4 == 0:
        Wt = W.t().contiguous()
        y.fill_(float("nan"))
        L.check(lib.fz_linear_forward_ex(x.data_ptr(), Wt.data_ptr(), b.data_ptr() if bias else None, y.data_ptr(), B, cin, cout, vox,
                                         0, 1, None, None, st))
        assert_close(_np(y), _np(ref), what="transposed weight")
    else:
        with pytest.raises(NotImplementedError):
            L.check(lib.fz_linear_forward_ex(x.data_ptr(), W.data_ptr(), None, y.data_ptr(), B, cin, cout, vox, 0, 1, None, None, st))
    with pytest.raises(ValueError):
        L.check(lib.fz_linear_forward_ex(x.data_ptr(), W.data_ptr(), None, y.data_ptr(), B, cin, cout, vox, 1, 0, None, None, st))
    assert not lib.fz_linear_forward_supported(cout, cin, vox + 2)
    assert not lib.fz_linear_forward_supported(cout, cin + 1, vox)


@pytest.mark.parametrize("nd,cin,cout,k,size,bias", [(3, 32, 64, 2, (32, 32, 32), True), (3, 4, 3, 1, (32, 32, 16), True),
                                                     (3, 24, 40, 2, (16, 32, 64), False), (2, 32, 64, 2, (128, 128), True),
                                                     (3, 8, 16, (2, 1, 2), (32, 16, 32), True), (3, 8, 8, 2, (12, 8, 6), True),
                                                     (3, 256, 512, 2, (16, 16, 16), True)])
def test_patch_convolution_as_channel_map(ft, dev, nd, cin, cout, k, size, bias):
    """ft.layers.ConvNd with kernel_size == stride (the reference U-Net's down-samplers and 1x1 head, unet.py:53,247)
    runs as a pointwise map on the space-to-depth view with the weight gradient from csrc/fz_linear.cu: output and
    all gradients against torch's own convolution in fp64; other shapes are the stock convolution."""
    from factorizer_b200 import layers
    torch.manual_seed(5)
    cls = getattr(layers, f"Conv{nd}d")
    conv = cls(cin, cout, kernel_size=k, stride=k, bias=bias).to(dev)
    x = torch.randn(2, cin, *size, device=dev, requires_grad=True)
    assert conv._patch_view(x) is not None
    y = conv(x)
    gy = torch.randn_like(y)
    params = [conv.weight] + ([conv.bias] if bias else [])
    grads = torch.autograd.grad((y * gy).sum(), [x] + params)
    fn = getattr(torch.nn.functional, f"conv{nd}d")
    x64 = x.detach().double().requires_grad_(True)
    p64 = [p.detach().double().requires_grad_(True) for p in params]
    y64 = fn(x64, p64[0], p64[1] if bias else None, stride=k)
    refs = torch.autograd.grad((y64 * gy.double()).sum(), [x64] + p64)
    assert y.shape == y64.shape
    assert_close(_np(y), _np(y64), what="y")
    for name, g, r in zip(["gx", "gw", "gb"], grads, refs):
        assert g.shape == r.shape
        scale = max(1.0, float(r.abs().max()))
        assert_close(_np(g) / scale, _np(r) / scale, what=name)
    # overlapping / padded convolutions are the library's; inference (no_grad) takes the same channel-map route
    assert cls(cin, cout, kernel_size=3, padding=1).to(dev)._patch_view(x) is None
    with torch.no_grad():
        assert conv._patch_view(x) is not None
        assert torch.equal(conv(x), y)


@pytest.mark.parametrize("nd,cin,cout,k,size,bias", [(3, 64, 32, 2, (16, 16, 16), True), (3, 40, 24, 2, (8, 16, 32), False),
                                                     (2, 64, 32, 2, (64, 64), True), (3, 16, 8, (2, 1, 2), (16, 16, 16), True),
                                                     (3, 8, 8, 2, (6, 4, 3), True), (3, 512, 256, 2, (8, 8, 8), True)])
def test_patch_transposed_convolution_as_channel_map(ft, dev, nd, cin, cout, k, size, bias):
    """ft.layers.ConvTransposeNd with kernel_size == stride (the reference U-Net's up-samplers, unet.py:97-99) as a
    pointwise map + depth-to-space: output and all gradients against torch's own transposed convolution in fp64."""
    from factorizer_b200 import layers
    torch.manual_seed(6)
    cls = getattr(layers, f"ConvTranspose{nd}d")
    conv = cls(cin, cout, kernel_size=k, stride=k, bias=bias).to(dev)
    x = torch.randn(2, cin, *size, device=dev, requires_grad=True)
    assert conv._patch_ok(x)
    y = conv(x)
    gy = torch.randn_like(y)
    params = [conv.weight] + ([conv.bias] if bias else [])
    grads = torch.autograd.grad((y * gy).sum(), [x] + params)
    fn = getattr(torch.nn.functional, f"conv_transpose{nd}d")
    x64 = x.detach().double().requires_grad_(True)
    p64 = [p.detach().double().requires_grad_(True) for p in params]
    y64 = fn(x64, p64[0], p64[1] if bias else None, stride=k)
    refs = torch.autograd.grad((y64 * gy.double()).sum(), [x64] + p64)
    assert y.shape == y64.shape
    assert_close(_np(y), _np(y64), what="y")
    for name, g, r in zip(["gx", "gw", "gb"], grads, refs):
        assert g.shape == r.shape
        scale = max(1.0, float(r.abs().max()))
        assert_close(_np(g) / scale, _np(r) / scale, what=name)
    assert not cls(cin, cout, kernel_size=3, stride=2).to(dev)._patch_ok(x)


@pytest.mark.parametrize("nd,cin,cout,k,pad,size,bias,xgrad", [(3, 4, 32, 3, 1, (32, 32, 32), False, False),
                                                               (3, 5, 12, (3, 1, 3), (1, 0, 1), (16, 16, 16), True, True),
                                                               (2, 3, 16, 5, 2, (64, 64), True, True),
                                                               (3, 2, 8, 3, 0, (18, 18, 18), True, False)])
def test_stem_convolution_weight_gradient(ft, dev, nd, cin, cout, k, pad, size, bias, xgrad):
    """ft.layers.ConvNd, stride 1 with few unfolded rows (the reference's 3x3x3 stem, factorizer.py:139-140): library
    forward / input gradient, weight gradient from csrc/fz_linear.cu on the unfolded input; against fp64 torch."""
    from factorizer_b200 import layers
    torch.manual_seed(7)
    cls = getattr(layers, f"Conv{nd}d")
    conv = cls(cin, cout, kernel_size=k, padding=pad, bias=bias).to(dev)
    x = torch.randn(2, cin, *size, device=dev, requires_grad=xgrad)
    assert conv._patch_view(x) is None and conv._unfold_ok(x)
    keep = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        y = conv(x)
        gy = torch.randn_like(y)
        params = [conv.weight] + ([conv.bias] if bias else [])
        wrt = ([x] if xgrad else []) + params
        grads = torch.autograd.grad((y * gy).sum(), wrt)
    finally:
        torch.backends.cudnn.allow_tf32 = keep
    fn = getattr(torch.nn.functional, f"conv{nd}d")
    x64 = x.detach().double().requires_grad_(xgrad)
    p64 = [p.detach().double().requires_grad_(True) for p in params]
    y64 = fn(x64, p64[0], p64[1] if bias else None, padding=pad)
    refs = torch.autograd.grad((y64 * gy.double()).sum(), ([x64] if xgrad else []) + p64)
    assert_close(_np(y), _np(y64), what="y")
    for i, (g, r) in enumerate(zip(grads, refs)):
        assert g.shape == r.shape
        scale = max(1.0, float(r.abs().max()))
        assert_close(_np(g) / scale, _np(r) / scale, what=f"grad {i}")
    assert not cls(64, 64, kernel_size=3, padding=1).to(dev)._unfold_ok(torch.randn(1, 64, 16, 16, 16, device=dev))
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():    # inference takes the same forward (direct kernel for the 3x3x3 -> 32 stem, library otherwise)
            assert_close(_np(conv(x)), _np(y64), what="no_grad y")
    finally:
        torch.backends.cudnn.allow_tf32 = keep


@pytest.mark.parametrize("cin,size,bias", [(4, (16, 12, 32), False), (1, (5, 7, 8), True), (3, (32, 32, 64), True), (2, (1, 1, 4), False)])
def test_stem_convolution_direct_kernel(ft, dev, cin, size, bias):
    """fz_conv3d_stem_forward (1..4 -> 32 channels, 3x3x3, padding 1) against torch's convolution in fp64, including
    volumes thinner than the kernel."""
    from factorizer_b200 import _ops
    torch.manual_seed(9)
    x = torch.randn(2, cin, *size, device=dev)
    w = torch.randn(32, cin, 3, 3, 3, device=dev) * 0.2
    b = torch.randn(32, device=dev) if bias else None
    assert _ops.stem_conv_supported(x, w, (1, 1, 1))
    y = _ops.conv3d_stem_forward(x, w, b)
    ref = torch.nn.functional.conv3d(x.double(), w.double(), None if b is None else b.double(), padding=1)
    assert_close(_np(y), _np(ref), what="y")
    assert not _ops.stem_conv_supported(torch.randn(1, 4, 8, 8, 6, device=dev), w[:, :4] if cin >= 4 else torch.randn(32, 4, 3, 3, 3, device=dev), (1, 1, 1))
    assert not _ops.stem_conv_supported(torch.randn(1, 8, 8, 8, 8, device=dev), torch.randn(32, 8, 3, 3, 3, device=dev), (1, 1, 1))


@pytest.mark.parametrize("shape", [(2, 3, 8, 6, 12), (1, 32, 32, 32, 32), (3, 1, 2, 2, 4)])
def test_space_to_depth_permutation(ft, dev, shape):
    """fz_space_depth2 against the einops-style permutation it replaces, both directions, bit-exact."""
    from factorizer_b200 import _ops
    torch.manual_seed(8)
    x = torch.randn(shape, device=dev)
    B, C, D, H, W = shape
    assert _ops.space_depth2_supported(x)
    ref = x.view(B, C, D // 2, 2, H // 2, 2, W // 2, 2).permute(0, 1, 3, 5, 7, 2, 4, 6).reshape(B, C * 8, -1)
    got = _ops.SpaceDepth2.apply(x, True, (D, H, W))
    assert torch.equal(got, ref)
    back = _ops.SpaceDepth2.apply(got, False, (D, H, W))
    assert torch.equal(back, x)
    xr = x.clone().requires_grad_(True)
    g = torch.randn_like(ref)
    (gx,) = torch.autograd.grad((_ops.SpaceDepth2.apply(xr, True, (D, H, W)) * g).sum(), xr)
    assert torch.equal(gx, _ops.SpaceDepth2.apply(g, False, (D, H, W)))
    assert not _ops.space_depth2_supported(torch.randn(1, 2, 4, 4, 6, device=dev))


def test_channel_map_layers_leave_autocast_to_the_library(ft, dev):
    """Under torch.autocast the fp32 channel-map kernels step aside: Linear and the patch / stem convolutions behave as
    the stock modules (reduced-precision output, working backward)."""
    from factorizer_b200 import layers
    torch.manual_seed(10)
    x = torch.randn(1, 32, 32, 32, 32, device=dev, requires_grad=True)
    mods = [ft.Linear(32, 64).to(dev), layers.Conv3d(32, 64, kernel_size=2, stride=2).to(dev),
            layers.ConvTranspose3d(32, 16, kernel_size=2, stride=2).to(dev)]
    stem = layers.Conv3d(4, 32, kernel_size=3, padding=1, bias=False).to(dev)
    x4 = torch.randn(1, 4, 32, 32, 32, device=dev)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        for m in mods:
            y = m(x)
            assert y.dtype == torch.bfloat16
            y.float().sum().backward()
            assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in m.parameters())
        assert stem._patch_view(x4) is None and not stem._unfold_ok(x4)
        y = stem(x4)
        assert y.dtype == torch.bfloat16
        y.float().sum().backward()
        assert torch.isfinite(stem.weight.grad).all()
    assert stem._unfold_ok(x4)


def test_layernorm_fallback_shapes(ft, dev):
    """Channel counts / voxel counts without a kernel take the reference's own permute + nn.LayerNorm route."""
    from factorizer_b200 import _ops
    x = torch.randn(2, 24, 5, 3, device=dev)          # odd number of voxels
    assert not _ops.layernorm_cf_supported(x)
    assert not _ops.layernorm_cf_supported(torch.randn(1, 600, 4, 4, device=dev))
    ln = ft.LayerNorm(24).to(dev)
    ref = torch.nn.functional.layer_norm(x.movedim(1, -1), (24,), ln.norm.weight, ln.norm.bias, ln.norm.eps).movedim(-1, 1)
    assert torch.allclose(ln(x), ref)


def test_saved_buffer_size_for_many_windows(ft, dev):
    """fz_swnmf_saved_bytes must size the buffer for the kernel family that runs: the octant kernels have no limit on the
    number of windows, the window-at-a-time kernels do (S * heads * g0 * g1 <= 4096).  A (1, 32, 8, 256, 256) volume has
    2 * 4 * 1 * 32 = 256 ... use a geometry beyond the limit: heads * g0 * g1 = 4 * 32 * 32 = 4096 per set."""
    import ctypes
    from factorizer_b200 import _lib, _ops
    shape = (1, 32, 256, 256, 8)
    sw = ft.SWMatricize((None, *shape[1:]), head_dim=8, patch_size=8)
    nmf = ft.NMF((8, 512), rank=1, num_iters=5, init="uniform", solver="hals").to(dev)
    g, s = sw._geom.c_geom(1), nmf.solver_spec().c_solver()
    need = _lib.lib().fz_swnmf_saved_bytes(ctypes.byref(g), ctypes.byref(s))
    assert need == 2 * 4 * 32 * 32 * 1 * (48 + 72) * 4
    x = torch.randn(shape, device=dev, requires_grad=True)
    y = _ops.SWNMF.apply(x, nmf.init.u0, nmf.init.v0, sw._geom, nmf.solver_spec(), True)
    (gx,) = torch.autograd.grad(y.sum(), x)          # used to fail with "saved buffer ... is required"
    assert torch.isfinite(gx).all()


def test_no_grad_inference_saves_nothing(ft, dev):
    """Under torch.no_grad() with parameters that require grad (inference with an unfrozen model) the fused ops must not
    allocate or fill the backward's buffers (ctx.needs_input_grad alone does not tell)."""
    from factorizer_b200 import _ops
    calls = []
    orig = _ops._swnmf_forward

    def spy(x, u0, v0, geom, spec, relu, need_grad):
        calls.append(need_grad)
        return orig(x, u0, v0, geom, spec, relu, need_grad)

    _ops._swnmf_forward = spy
    try:
        blk = ft.FactorizerBlock(channels=32, spatial_size=(16, 16, 16), norm=ft.LayerNorm,
                                 reshape=(ft.SWMatricize, {"head_dim": 8, "patch_size": 8}), act=nn.ReLU, factorize=ft.NMF,
                                 rank=1, num_iters=5, init="uniform", solver="hals", mlp_ratio=2, dropout=0.0).to(dev)
        x = torch.randn(1, 32, 16, 16, 16, device=dev)
        with torch.no_grad():
            blk(x)
        blk(x)
    finally:
        _ops._swnmf_forward = orig
    assert calls == [False, True]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_two_devices_in_one_process(ft):
    """cudaFuncSetAttribute (dynamic shared memory above 48 KiB) and the SM count are per device: the second GPU of a
    process must work like the first (the octant kernels use 192-224 KiB)."""
    from factorizer_b200 import _ops
    outs = []
    for d in (0, 1):
        dev = torch.device("cuda", d)
        sw = ft.SWMatricize((None, 8, 16, 16, 16), head_dim=8, patch_size=8)
        torch.manual_seed(0)
        nmf = ft.NMF((8, 512), rank=1, num_iters=5, init="uniform", solver="hals").to(dev)
        torch.manual_seed(1)
        x = torch.randn(1, 8, 16, 16, 16).to(dev).requires_grad_(True)
        with torch.cuda.device(dev):
            y = _ops.SWNMF.apply(x, nmf.init.u0, nmf.init.v0, sw._geom, nmf.solver_spec(), True)
            (gx,) = torch.autograd.grad(y.sum(), x)
        outs.append((y.detach().cpu(), gx.cpu()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
