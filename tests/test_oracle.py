"""The numpy oracle (oracle/factorizer_oracle.py) pinned against golden vectors produced by the
reference itself (tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest

import cases
from conftest import assert_close, tol_ratio
from oracle import factorizer_oracle as O


def _geom(c):
    xs = c["x_shape"]
    n = len(xs) - 2
    kw = dict(c["kw"])
    shifts = kw.pop("shifts", None)
    H, d, grid, patch = O.resolve_geometry((None, *xs[1:]), **kw)
    if c["cls"] == "SWMatricize":
        shifts = O.default_shifts(patch) if shifts is None else shifts
    else:
        shifts = [shifts]
    return H, d, grid, patch, O.normalise_shifts(shifts, n)


@pytest.mark.parametrize("name", list(cases.SW_CASES))
def test_swmat_bit_exact(golden, name):
    c = cases.SW_CASES[name]
    g = golden["sw"]
    H, d, grid, patch, shifts = _geom(c)
    x = cases.make_array(name, c["x_shape"], "randn")
    y = O.swmat_forward(x, H, d, grid, patch, shifts)
    assert tuple(g[f"{name}/y_shape"]) == y.shape
    assert cases.digest(y) == str(g[f"{name}/y_digest"])
    w = cases.make_array(name, y.shape, "randn", tag="w")
    z = O.swmat_inverse(w, x.shape[0], H, d, grid, patch, shifts)
    assert cases.digest(z) == str(g[f"{name}/z_digest"])
    rt = O.swmat_inverse(y, x.shape[0], H, d, grid, patch, shifts)
    assert cases.digest(rt) == str(g[f"{name}/rt_digest"])
    assert bool(g[f"{name}/roundtrip_equal"]) == bool(np.array_equal(rt, x))


# HALS with rank >= 2 is ill-conditioned in the reference itself (SURVEY App. C): a ReLU-mask flip
# between two fp32 evaluation orders changes the gradient.  Those cases are compared to the fp64
# reference with the bound the fp32 reference itself achieves.
WELL_CONDITIONED = {n for n, c in cases.NMF_CASES.items() if c["solver"] == "mu" or c["rank"] == 1}


@pytest.mark.parametrize("name", list(cases.NMF_CASES))
def test_nmf_forward_backward(golden, name):
    c = cases.NMF_CASES[name]
    g = golden["nmf"]
    x = cases.make_array(name, c["shape"], c["dist"])
    gy = cases.make_array(name, c["shape"], "randn", tag="gy")
    u0, v0 = g[f"{name}/u0"], g[f"{name}/v0"]
    u, v = O.nmf_decompose(x, u0, v0, c["solver"], c["num_iters"])
    y = O.nmf_forward(x, u0, v0, c["solver"], c["num_iters"])
    gx = O.nmf_backward(x, u0, v0, gy=gy, solver=c["solver"], num_iters=c["num_iters"],
                        num_grad_steps=c["num_grad_steps"])
    assert (u >= 0).all() and (v >= 0).all()      # reference tests/test_nmf.py:19-20
    if name in WELL_CONDITIONED:
        assert_close(u, g[f"{name}/u"], what="u")
        assert_close(v, g[f"{name}/v"], what="v")
        assert_close(y, g[f"{name}/y"], what="y")
        assert_close(gx, g[f"{name}/gx"], what="gx")
    else:
        ref_gap = max(tol_ratio(g[f"{name}/y"], g[f"{name}/y64"]), tol_ratio(g[f"{name}/gx"], g[f"{name}/gx64"]))
        ours = max(tol_ratio(y, g[f"{name}/y64"]), tol_ratio(gx, g[f"{name}/gx64"]))
        assert ours <= max(1.0, 10 * ref_gap), (ours, ref_gap)


@pytest.mark.parametrize("name", list(cases.NMF_CASES))
def test_nmf_fp64_matches_reference_fp64(golden, name):
    """In float64 the oracle's hand-derived adjoint must agree with the reference's autograd to
    rounding, whatever the conditioning."""
    c = cases.NMF_CASES[name]
    g = golden["nmf"]
    x = cases.make_array(name, c["shape"], c["dist"]).astype(np.float64)
    gy = cases.make_array(name, c["shape"], "randn", tag="gy").astype(np.float64)
    u0, v0 = g[f"{name}/u0"].astype(np.float64), g[f"{name}/v0"].astype(np.float64)
    y = O.nmf_forward(x, u0, v0, c["solver"], c["num_iters"])
    gx = O.nmf_backward(x, u0, v0, gy=gy, solver=c["solver"], num_iters=c["num_iters"],
                        num_grad_steps=c["num_grad_steps"])
    assert_close(y, g[f"{name}/y64"], rtol=1e-9, atol=1e-11, what="y64")
    scale = max(1.0, float(np.abs(g[f"{name}/gx64"]).max()))
    assert_close(gx / scale, g[f"{name}/gx64"] / scale, rtol=1e-7, atol=1e-9, what="gx64")


@pytest.mark.parametrize("name", list(cases.FUSED_CASES))
def test_fused_core(golden, name):
    c = cases.FUSED_CASES[name]
    g = golden["fused"]
    H, d, grid, patch, shifts = _geom(c)
    x = cases.make_array(name, c["x_shape"], c["dist"])
    gy = cases.make_array(name, c["x_shape"], "randn", tag="gy")
    u0, v0 = g[f"{name}/u0"], g[f"{name}/v0"]
    nm = c["nmf"]
    y = O.swnmf_forward(x, u0, v0, H, d, grid, patch, shifts, relu=c["relu"], solver=nm["solver"],
                        num_iters=nm["num_iters"])
    gx = O.swnmf_backward(x, gy, u0, v0, H, d, grid, patch, shifts, relu=c["relu"], solver=nm["solver"],
                          num_iters=nm["num_iters"], num_grad_steps=nm.get("num_grad_steps"))
    assert_close(y, g[f"{name}/y"], what="y")
    assert_close(gx, g[f"{name}/gx"], what="gx")


C_CASES = [n for n, c in cases.FUSED_CASES.items()
           if c["nmf"]["solver"] == "hals" and c["nmf"]["rank"] == 1 and len(c["x_shape"]) == 5]


@pytest.mark.parametrize("name", C_CASES)
def test_c_oracle_matches_golden(golden, name):
    """oracle/nmf_oracle.c (the OpenMP CPU baseline) against the reference's outputs."""
    from oracle import c_oracle
    c = cases.FUSED_CASES[name]
    g = golden["fused"]
    H, d, grid, patch, shifts = _geom(c)
    x = cases.make_array(name, c["x_shape"], c["dist"])
    gy = cases.make_array(name, c["x_shape"], "randn", tag="gy")
    nm = c["nmf"]
    y = c_oracle.swnmf_forward(x, g[f"{name}/v0"], d, patch, shifts, relu=c["relu"], num_iters=nm["num_iters"])
    gx = c_oracle.swnmf_backward(x, gy, g[f"{name}/v0"], d, patch, shifts, relu=c["relu"],
                                 num_iters=nm["num_iters"], num_grad_steps=nm.get("num_grad_steps"))
    assert_close(y, g[f"{name}/y"], what="y")
    assert_close(gx, g[f"{name}/gx"], what="gx")


@pytest.mark.parametrize("name", ["hals_r1_8x512", "hals_r1_relu_randn", "hals_r1_zero_window", "hals_r1_8x64_T3_k1",
                                  "hals_r1_32x64"])
def test_gram_form_is_well_conditioned(golden, name):
    """The Gram-matrix form the CUDA kernels evaluate for act = ReLU (csrc/fz_swnmf_gram.cuh) equals the
    reference's unrolled solver: exactly in fp64, and in fp32 no further from the fp64 reference than
    the reference's own fp32 run is (plus a small slack)."""
    c = cases.NMF_CASES[name]
    g = golden["nmf"]
    M, N = c["shape"][-2:]
    x = cases.make_array(name, c["shape"], c["dist"]).reshape(-1, M, N)
    gy = cases.make_array(name, c["shape"], "randn", tag="gy").reshape(-1, M, N)
    v0 = g[f"{name}/v0"][:, 0]
    kw = dict(num_iters=c["num_iters"], num_grad_steps=c["num_grad_steps"])
    y64, gx64 = g[f"{name}/y64"], g[f"{name}/gx64"]
    yr, gr = g[f"{name}/y"], g[f"{name}/gx"]
    y, dx = (a.reshape(c["shape"]) for a in O.hals_r1_gram(x.astype(np.float64), v0.astype(np.float64), gy.astype(np.float64), **kw))
    assert tol_ratio(y, y64) < 1e-6 and tol_ratio(dx, gx64) < 1e-6
    y, dx = (a.reshape(c["shape"]) for a in O.hals_r1_gram(x, v0, gy, **kw))
    assert_close(y, yr, what="y")
    assert_close(dx, gr, what="gx")
    assert tol_ratio(y, y64) <= tol_ratio(yr, y64) + 0.02
    assert tol_ratio(dx, gx64) <= tol_ratio(gr, gx64) + 0.05


@pytest.mark.parametrize("name", list(cases.BLOCK_CASES))
def test_oracle_block_matches_reference(golden, name):
    """FactorizerBlock glue of the oracle (LayerNorm / Linear / GELU MLP / residuals around the core), forward
    and hand-derived backward, against the reference's own forward + autograd (block.npz); fp64 arithmetic
    on the fp32 inputs, so the bound is the reference's fp32 rounding."""
    c, g = cases.BLOCK_CASES[name], golden["block"]
    sd = {k.split("/sd/")[1]: g[k].astype(np.float64) for k in g if k.startswith(name + "/sd/")}
    xs = (c["batch"], c["channels"], *c["spatial"])
    x = cases.make_array(name, xs, "randn").astype(np.float64)
    gy = cases.make_array(name, xs, "randn", tag="gy").astype(np.float64)
    H, d, grid, patch = O.resolve_geometry((None, *xs[1:]), **c["kw"])
    shifts = O.normalise_shifts(O.default_shifts(patch), len(patch))
    y = O.block_forward(x, sd, H, d, grid, patch, shifts)
    gx, gp = O.block_backward(x, gy, sd, H, d, grid, patch, shifts)
    assert_close(y, g[f"{name}/y"], what="y")
    assert_close(gx, g[f"{name}/gx"], what="gx")
    for k, v in gp.items():
        ref = g[f"{name}/gp/{k}"]
        scale = max(1.0, float(np.abs(ref).max()))
        assert_close(v / scale, ref / scale, rtol=1e-4, atol=1e-4, what=f"grad {k}")


@pytest.mark.parametrize("name", ["block_c16_16", "block_c32_16"])
def test_torch_port_matches_golden(golden, name):
    """oracle/torch_port.py (the CPU baseline bench.py times: the reference's ATen operator sequence restated in plain
    torch, differentiated by autograd) against the reference's own outputs and gradients for a FactorizerBlock."""
    import torch
    from oracle import torch_port as TP
    c, g = cases.BLOCK_CASES[name], golden["block"]
    sd = {k.split("/sd/")[1]: torch.from_numpy(g[k]).requires_grad_(True) for k in g if k.startswith(name + "/sd/")}
    xs = (c["batch"], c["channels"], *c["spatial"])
    x = torch.from_numpy(cases.make_array(name, xs, "randn")).requires_grad_(True)
    gy = torch.from_numpy(cases.make_array(name, xs, "randn", tag="gy"))
    y = TP.block_forward(x, sd)
    names = [k for k in sd if not k.endswith(("u0", "v0"))]
    grads = torch.autograd.grad((y * gy).sum(), [x] + [sd[k] for k in names])
    assert_close(y.detach().numpy(), g[f"{name}/y"], what="y")
    assert_close(grads[0].numpy(), g[f"{name}/gx"], what="gx")
    for k, gp in zip(names, grads[1:]):
        ref = g[f"{name}/gp/{k}"]
        scale = max(1.0, float(np.abs(ref).max()))
        assert_close(gp.numpy() / scale, ref / scale, rtol=1e-4, atol=1e-4, what=f"grad {k}")
