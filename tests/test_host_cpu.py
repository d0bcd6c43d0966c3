"""CPU-only checks: the C-ABI library loads and exports every symbol the header declares, the host
modules mirror the reference's constructor / state_dict contract, and the product path refuses to
run without CUDA (no fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch
from torch import nn

import cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ft():
    from factorizer_b200 import _build
    _build.build()
    import factorizer_b200
    return factorizer_b200


def test_library_exports_every_declared_symbol(ft):
    from factorizer_b200 import _lib
    header = open(os.path.join(ROOT, "include", "factorizer_b200.h")).read()
    declared = set(re.findall(r"\b(fz_[a-z_0-9]+)\s*\(", header))
    declared -= {"fz_geom", "fz_solver"}
    handle = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in the header but not exported"
    assert declared == set(_lib.exported_symbols())
    assert _lib.lib().fz_version() == 100


def test_struct_layout_matches_header(ft):
    from factorizer_b200 import _lib
    assert ctypes.sizeof(_lib.FzGeom) == 4 * (2 + 3 + 3 + 2 + 3 * 8 + 2)
    assert ctypes.sizeof(_lib.FzSolver) == 20


def test_geometry_validation_through_abi(ft):
    from factorizer_b200 import _lib
    lib = _lib.lib()
    g = _lib.make_geom(1, 32, (16, 16, 16), (8, 8, 5), 8, [(0, 0, 0)])
    s = _lib.make_solver(_lib.FZ_SOLVER_HALS, 1, 5, 5, 1e-16)
    # size not divisible by patch -> invalid geometry -> 0 bytes, and the entry point reports it
    assert lib.fz_swnmf_saved_bytes(ctypes.byref(g), ctypes.byref(s)) == 0
    code = lib.fz_swmat_forward(None, None, ctypes.byref(g), None)
    assert code == _lib.FZ_ERR_INVALID
    assert b"divisible" in lib.fz_last_error()
    s2 = _lib.make_solver(7, 1, 5, 5, 1e-16)
    code = lib.fz_nmf_forward(None, None, None, None, None, None, 1, 8, 16, ctypes.byref(s2), None)
    assert code == _lib.FZ_ERR_UNSUPPORTED


def test_channel_map_epilogue_arguments_through_abi(ft):
    """Return codes of the two channel-map entries on bad epilogue arguments (refused before any device work).  The fp32
    entry rejects an unknown epilogue even for a zero batch; the bf16 entry returns early on a zero batch."""
    from factorizer_b200 import _lib
    lib = _lib.lib()
    p = 256                                       # a non-null address the refused calls never dereference
    fwd = lambda batch, epi, aux, y2: lib.fz_linear_forward_ex(p, p, None, p, batch, 8, 8, 64, epi, 0, aux, y2, None)
    bf16 = lambda batch, epi, aux, y2: lib.fz_linear_forward_bf16(p, p, 8, None, p, batch, 8, 8, 64, epi, aux, y2, None)
    assert fwd(0, 7, p, p) == _lib.FZ_ERR_INVALID
    assert fwd(0, -1, p, p) == _lib.FZ_ERR_INVALID
    assert fwd(0, 1, None, None) == _lib.FZ_OK
    assert fwd(1, 7, p, p) == _lib.FZ_ERR_INVALID
    assert fwd(1, 1, None, p) == _lib.FZ_ERR_INVALID
    assert fwd(1, 3, None, p) == _lib.FZ_ERR_INVALID
    assert fwd(1, 2, p, None) == _lib.FZ_ERR_INVALID
    assert bf16(0, 7, None, None) == _lib.FZ_OK
    assert bf16(1, 7, p, p) == _lib.FZ_ERR_INVALID
    assert bf16(1, 1, None, p) == _lib.FZ_ERR_INVALID
    assert bf16(1, 3, None, p) == _lib.FZ_ERR_INVALID
    assert bf16(1, 2, p, None) == _lib.FZ_ERR_INVALID


def test_readme_shapes_and_state_dict_keys(ft, golden):
    sw = ft.SWMatricize((None, 32, 128, 128, 128), head_dim=8, patch_size=8)
    assert sw.output_size == (None, 4096, 8, 512)          # reference README.md:43-47
    assert len(sw.shifted_windows) == 2
    assert not hasattr(sw.shifted_windows[0], "shifts")    # reference operations.py:191-194
    assert sw.shifted_windows[1].shifts == (4, 4, 4) and sw.shifted_windows[1].dims == (2, 3, 4)
    c = cases.BLOCK_CASES["block_c16_16"]
    blk = ft.FactorizerBlock(channels=c["channels"], spatial_size=c["spatial"], norm=ft.LayerNorm,
                             reshape=(ft.SWMatricize, c["kw"]), act=nn.ReLU, factorize=ft.NMF,
                             mlp_ratio=c["mlp_ratio"], dropout=0.0, **c["nmf"])
    ref_keys = [k.split("/sd/")[1] for k in golden["block"] if k.startswith("block_c16_16/sd/")]
    assert list(blk.state_dict().keys()) == ref_keys
    for k, v in blk.state_dict().items():
        assert tuple(v.shape) == golden["block"][f"block_c16_16/sd/{k}"].shape


def _build_model(ft, c):
    return ft.Factorizer(in_channels=c["in_channels"], out_channels=c["out_channels"], spatial_size=c["spatial"],
                         norm=ft.LayerNorm, reshape=(ft.SWMatricize, c["reshape_kw"]), act=nn.ReLU, factorize=ft.NMF,
                         **c["kw"])


@pytest.mark.parametrize("name", list(cases.MODEL_CASES))
def test_factorizer_model_state_dict_matches_reference(ft, golden, name):
    """ft.Factorizer (reference factorizer/factorizer.py:125-171 on unet.py:177-276): same module tree, hence the
    same state_dict keys in the same order and the same shapes, and the same consumption of the global RNG at
    construction (every buffer / parameter drawn before the generator's perturbation is bit-identical)."""
    c, g = cases.MODEL_CASES[name], golden["model"]
    torch.manual_seed(cases._seed(name) % (2**31))
    net = _build_model(ft, c)
    ref_keys = [k.split("/sd/")[1] for k in g if k.startswith(name + "/sd/")]
    sd = net.state_dict()
    assert list(sd.keys()) == ref_keys
    for k, v in sd.items():
        ref = g[f"{name}/sd/{k}"]
        assert tuple(v.shape) == ref.shape
        if v.ndim != 1:   # 1-D parameters were perturbed after construction by make_golden.py
            np.testing.assert_array_equal(v.numpy(), ref, err_msg=k)
    net.load_state_dict({k: torch.from_numpy(g[f"{name}/sd/{k}"]) for k in ref_keys})
    # deep supervision heads (unet.py:252-259, 269-276)
    net2 = ft.Factorizer(in_channels=1, out_channels=2, spatial_size=(16, 16), encoder_depth=(1, 1, 1),
                         encoder_width=(8, 16, 32), strides=(1, 2, 2), decoder_depth=(1, 1), num_deep_supr=2,
                         reshape=(ft.SWMatricize, {"head_dim": 4, "patch_size": 4}), rank=1)
    assert [k for k in net2.state_dict() if k.startswith("head")] == ["heads.0.weight", "heads.0.bias", "heads.1.weight",
                                                                     "heads.1.bias"]
    with pytest.raises(NotImplementedError):
        ft.UNet(1, 2)


@pytest.mark.parametrize("name", list(cases.SW_CASES))
def test_output_size_matches_reference(ft, golden, name):
    c = cases.SW_CASES[name]
    mod = getattr(ft, c["cls"])((None, *c["x_shape"][1:]), **c["kw"])
    want = tuple(None if v < 0 else int(v) for v in golden["sw"][f"{name}/output_size"])
    assert tuple(mod.output_size) == want


def test_random_init_consumes_rng_like_reference(ft, golden):
    # same seed -> same u0/v0 as the reference drew (u0 first, then v0; matrix_factorization.py:44-50)
    name = "cfg1_mu_r2"
    torch.manual_seed(cases._seed(name) % (2**31))
    nmf = ft.NMF(size=(8, 512), rank=2, num_iters=5, init="uniform", solver="mu")
    np.testing.assert_array_equal(nmf.init.u0.numpy(), golden["nmf"][f"{name}/u0"])
    np.testing.assert_array_equal(nmf.init.v0.numpy(), golden["nmf"][f"{name}/v0"])


def test_rank_from_compression(ft):
    assert ft.NMF(size=(8, 512)).rank == 1                  # ceil(4096 / (10*520)) = 1
    assert ft.NMF(size=(32, 64)).rank == 3
    assert ft.NMF(size=(8, 16), rank=3).compression == pytest.approx(8 * 16 / (3 * 24))


def test_out_of_scope_names_raise(ft):
    for spec in ("cd", "ls", "fmu", "smu", "mu-0"):
        with pytest.raises(NotImplementedError):
            ft.NMF(size=(8, 16), solver=spec)
    with pytest.raises(NotImplementedError):
        ft.NMF(size=(8, 16), init="svd")
    with pytest.raises(NotImplementedError):
        ft.MatrixFactorization(size=(8, 16))                # reference default solver 'cd'
    assert ft.NMF(size=(64, 512)).rank == 6                 # the default compression on a 64 x 512 matrix: within FZ_MAX_RANK = 8
    with pytest.raises(NotImplementedError):
        ft.NMF(size=(16, 32), rank=9)


def test_no_cpu_fallback(ft):
    nmf = ft.NMF(size=(8, 16), rank=1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        nmf(torch.rand(2, 8, 16))
    sw = ft.SWMatricize((None, 8, 8, 8, 8), head_dim=8, patch_size=4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        sw(torch.rand(1, 8, 8, 8, 8))


def test_product_does_not_import_oracle():
    """The oracle is test infrastructure: nothing under factorizer_b200/ may import or execute it."""
    pkg = os.path.join(ROOT, "factorizer_b200")
    pat = re.compile(r"^\s*(from|import)\s+oracle|oracle[/.]factorizer_oracle|importlib.*oracle", re.M)
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not pat.search(src), f


def test_deep_supervision_heads_follow_the_reference(ft):
    """factorizer/unet.py:251-258: `num_deep_supr=True` stores 3 but builds range(True) = ONE head; an int n builds n.
    The module tree (state_dict keys heads.0 ...) must agree or reference checkpoints do not load."""
    kw = dict(in_channels=1, out_channels=2, spatial_size=(16, 16, 16), encoder_depth=(1, 1), encoder_width=(8, 16), strides=(1, 2),
              decoder_depth=(1,), norm=ft.LayerNorm, reshape=(ft.SWMatricize, {"head_dim": 8, "patch_size": 8}), act=nn.ReLU,
              factorize=ft.NMF, rank=1, num_iters=2, init="uniform", solver="hals", mlp_ratio=2)
    net = ft.Factorizer(num_deep_supr=True, **kw)
    assert len(net.heads) == 1 and net.num_deep_supr == 3
    assert [k for k in net.state_dict() if k.startswith("heads.")][0].startswith("heads.0.")
    assert len(ft.Factorizer(num_deep_supr=2, **kw).heads) == 2
    assert hasattr(ft.Factorizer(num_deep_supr=False, **kw), "head")
