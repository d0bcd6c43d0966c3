"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED reference
(pashtari/factorizer, /root/reference) on the seeded inputs of cases.py.

Build-container only (the reference does not exist on the GPU box):

    python tests/golden/make_golden.py

The reference imports ``opt_einsum`` (factorizer/factorization/matrix_factorization.py:8) but never
uses it; an empty stub module stands in for it.  Outputs: nmf.npz, sw.npz, fused.npz, block.npz, model.npz
(cases.save_golden: the outputs of the larger cases at a seeded sample of indices, each file below 1 MB).
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.modules.setdefault("opt_einsum", types.ModuleType("opt_einsum"))
sys.path.insert(0, os.environ.get("FZ_REFERENCE", "/root/reference"))

import factorizer as ft  # noqa: E402  (the reference)
from torch import nn  # noqa: E402

import cases  # noqa: E402

torch.set_num_threads(4)


def t(a):
    return torch.from_numpy(a.copy())


def gen_nmf():
    out = {}
    for name, c in cases.NMF_CASES.items():
        torch.manual_seed(cases._seed(name) % (2**31))
        M, N = c["shape"][-2:]
        nmf = ft.NMF(size=(M, N), rank=c["rank"], num_iters=c["num_iters"],
                     num_grad_steps=c["num_grad_steps"], init="uniform", solver=c["solver"])
        x = t(cases.make_array(name, c["shape"], c["dist"])).requires_grad_(True)
        gy = t(cases.make_array(name, c["shape"], "randn", tag="gy"))
        u, v = nmf.decompose(x)
        y = nmf.reconstruct(u, v)
        (gx,) = torch.autograd.grad((y * gy).sum(), x)
        out[f"{name}/u0"] = nmf.init.u0.numpy().copy()
        out[f"{name}/v0"] = nmf.init.v0.numpy().copy()
        out[f"{name}/u"] = u.detach().numpy()
        out[f"{name}/v"] = v.detach().numpy()
        out[f"{name}/y"] = y.detach().numpy()
        out[f"{name}/gx"] = gx.numpy()
        # float64 run of the reference itself: separates "we differ" from "fp32 is ill-conditioned"
        nmf64 = ft.NMF(size=(M, N), rank=c["rank"], num_iters=c["num_iters"],
                       num_grad_steps=c["num_grad_steps"], init="uniform", solver=c["solver"]).double()
        nmf64.init.u0.copy_(nmf.init.u0.double())
        nmf64.init.v0.copy_(nmf.init.v0.double())
        x64 = x.detach().double().requires_grad_(True)
        y64 = nmf64(x64)
        (gx64,) = torch.autograd.grad((y64 * gy.double()).sum(), x64)
        out[f"{name}/y64"] = y64.detach().numpy()
        out[f"{name}/gx64"] = gx64.numpy()
    cases.save_golden(HERE, "nmf", out)
    print("nmf.npz", len(out), "arrays")


def gen_sw():
    out = {}
    for name, c in cases.SW_CASES.items():
        xs = c["x_shape"]
        mod = getattr(ft, c["cls"])((None, *xs[1:]), **c["kw"])
        x = t(cases.make_array(name, xs, "randn"))
        y = mod(x)
        out[f"{name}/y_shape"] = np.array(y.shape, dtype=np.int64)
        out[f"{name}/y_digest"] = np.array(cases.digest(y.numpy()))
        out[f"{name}/output_size"] = np.array([-1 if s is None else s for s in mod.output_size], dtype=np.int64)
        # a few samples for debugging index maps
        flat = y.numpy().reshape(-1)
        idx = np.random.Generator(np.random.PCG64(1)).integers(0, flat.size, 64)
        out[f"{name}/y_idx"] = idx
        out[f"{name}/y_val"] = flat[idx]
        # inverse on an independent random matricised tensor (not a round trip)
        w = t(cases.make_array(name, tuple(y.shape), "randn", tag="w"))
        z = mod.inverse_forward(w)
        out[f"{name}/z_digest"] = np.array(cases.digest(z.numpy()))
        out[f"{name}/z"] = z.numpy() if z.numel() <= 16384 else z.numpy().reshape(-1)[:16384]
        # README.md:49-51 round trip
        rt = mod.inverse_forward(y)
        out[f"{name}/roundtrip_equal"] = np.array(bool(torch.equal(rt, x)))
        out[f"{name}/rt_digest"] = np.array(cases.digest(rt.numpy()))
    cases.save_golden(HERE, "sw", out)
    print("sw.npz", len(out), "arrays")


def gen_fused():
    out = {}
    for name, c in cases.FUSED_CASES.items():
        torch.manual_seed(cases._seed(name) % (2**31))
        xs = c["x_shape"]
        reshape = getattr(ft, c["cls"])((None, *xs[1:]), **c["kw"])
        nmf = ft.NMF(reshape.output_size[2:], init="uniform", **c["nmf"])
        x = t(cases.make_array(name, xs, c["dist"])).requires_grad_(True)
        gy = t(cases.make_array(name, xs, "randn", tag="gy"))
        # FactMixer.forward core, factorizer/factorizer.py:41-50
        m = reshape(x)
        if c["relu"]:
            m = torch.relu(m)
        m = nmf(m)
        y = reshape.inverse_forward(m)
        (gx,) = torch.autograd.grad((y * gy).sum(), x)
        out[f"{name}/u0"] = nmf.init.u0.numpy().copy()
        out[f"{name}/v0"] = nmf.init.v0.numpy().copy()
        out[f"{name}/y"] = y.detach().numpy()
        out[f"{name}/gx"] = gx.numpy()
    cases.save_golden(HERE, "fused", out)
    print("fused.npz", len(out), "arrays")


def gen_block():
    out = {}
    for name, c in cases.BLOCK_CASES.items():
        torch.manual_seed(cases._seed(name) % (2**31))
        blk = ft.FactorizerBlock(
            channels=c["channels"], spatial_size=c["spatial"], norm=ft.LayerNorm,
            reshape=(ft.SWMatricize, c["kw"]), act=nn.ReLU, factorize=ft.NMF,
            mlp_ratio=c["mlp_ratio"], dropout=0.0, **c["nmf"])
        # perturb LayerNorm affine params so they are not the identity
        with torch.no_grad():
            for p in blk.parameters():
                if p.ndim == 1:
                    p.add_(0.1 * torch.randn_like(p))
        xs = (c["batch"], c["channels"], *c["spatial"])
        x = t(cases.make_array(name, xs, "randn")).requires_grad_(True)
        gy = t(cases.make_array(name, xs, "randn", tag="gy"))
        y = blk(x)
        params = list(blk.parameters())
        grads = torch.autograd.grad((y * gy).sum(), [x] + params)
        for k, v in blk.state_dict().items():
            out[f"{name}/sd/{k}"] = v.numpy().copy()
        out[f"{name}/y"] = y.detach().numpy()
        out[f"{name}/gx"] = grads[0].numpy()
        for (k, _), g in zip(blk.named_parameters(), grads[1:]):
            out[f"{name}/gp/{k}"] = g.numpy()
    cases.save_golden(HERE, "block", out)
    print("block.npz", len(out), "arrays")


def gen_model():
    out = {}
    for name, c in cases.MODEL_CASES.items():
        torch.manual_seed(cases._seed(name) % (2**31))
        net = ft.Factorizer(in_channels=c["in_channels"], out_channels=c["out_channels"], spatial_size=c["spatial"],
                            norm=ft.LayerNorm, reshape=(ft.SWMatricize, c["reshape_kw"]), act=nn.ReLU,
                            factorize=ft.NMF, **c["kw"]).eval()
        with torch.no_grad():
            for p in net.parameters():
                if p.ndim == 1:
                    p.add_(0.1 * torch.randn_like(p))
        xs = (c["batch"], c["in_channels"], *c["spatial"])
        x = t(cases.make_array(name, xs, "randn")).requires_grad_(True)
        y = net(x)
        gy = t(cases.make_array(name, tuple(y.shape), "randn", tag="gy"))
        params = list(net.parameters())
        grads = torch.autograd.grad((y * gy).sum(), [x] + params)
        for k, v in net.state_dict().items():
            out[f"{name}/sd/{k}"] = v.numpy().copy()
        out[f"{name}/y"] = y.detach().numpy()
        out[f"{name}/gx"] = grads[0].numpy()
        for (k, _), g in zip(net.named_parameters(), grads[1:]):
            out[f"{name}/gp/{k}"] = g.numpy()
    cases.save_golden(HERE, "model", out)
    print("model.npz", len(out), "arrays")


if __name__ == "__main__":
    gen_nmf()
    gen_sw()
    gen_fused()
    gen_block()
    gen_model()
