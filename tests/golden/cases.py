"""Seeded case definitions shared by the golden-vector generator (make_golden.py, which runs the
reference in the build container) and by the tests (which re-create the same inputs and compare
against the committed outputs).  Inputs come from numpy's PCG64 so they are identical everywhere;
only the reference's *outputs* (and its torch-RNG-initialised u0/v0 buffers) live in the .npz files.
"""
from __future__ import annotations

import hashlib
import os

import numpy as np

# --- plain NMF on already-matricised tensors (ft.NMF.forward / decompose) ------------------------
# name -> dict(shape, rank, solver, num_iters, num_grad_steps, dist)
NMF_CASES = {
    # BASELINE config 1 / README.md:34-38
    "cfg1_mu_r2": dict(shape=(1, 8, 512), rank=2, solver="mu", num_iters=5, num_grad_steps=None, dist="uniform"),
    "hals_r1_8x512": dict(shape=(4, 3, 8, 512), rank=1, solver="hals", num_iters=5, num_grad_steps=None, dist="uniform"),
    "hals_r1_relu_randn": dict(shape=(6, 8, 512), rank=1, solver="hals", num_iters=5, num_grad_steps=None, dist="relu_randn"),
    # reference tests/test_nmf.py:9-12
    "hals_r3_8x16": dict(shape=(2, 4, 8, 16), rank=3, solver="hals", num_iters=5, num_grad_steps=None, dist="uniform"),
    "mu_r1_16x64": dict(shape=(5, 16, 64), rank=1, solver="mu", num_iters=5, num_grad_steps=None, dist="uniform"),
    "hals_r2_4x64_k2": dict(shape=(3, 4, 64), rank=2, solver="hals", num_iters=5, num_grad_steps=2, dist="uniform"),
    "hals_r1_8x64_T3_k1": dict(shape=(7, 8, 64), rank=1, solver="hals", num_iters=3, num_grad_steps=1, dist="uniform"),
    "hals_r1_zero_window": dict(shape=(3, 8, 512), rank=1, solver="hals", num_iters=5, num_grad_steps=None, dist="zero_first"),
    "mu_r2_32x64": dict(shape=(4, 32, 64), rank=2, solver="mu", num_iters=4, num_grad_steps=None, dist="uniform"),
    "hals_r1_32x64": dict(shape=(2, 3, 32, 64), rank=1, solver="hals", num_iters=5, num_grad_steps=None, dist="uniform"),
    # ranks above 4: ft.NMF((64, 512)) with the reference's default compression=10 resolves to rank 6
    # (matrix_factorization.py:480-487); rank 8 is FZ_MAX_RANK
    # (at 64 x 512 the backward's working set exceeds one CTA's shared memory, at 128 x 1024 the forward's too: X and dX stay in
    # global memory there, csrc/fz_nmf_generic.cu `spill`)
    "mu_r6_64x512": dict(shape=(1, 64, 512), rank=6, solver="mu", num_iters=5, num_grad_steps=None, dist="uniform"),
    "mu_r2_128x1024": dict(shape=(1, 128, 1024), rank=2, solver="mu", num_iters=4, num_grad_steps=None, dist="uniform"),
    "mu_r6_32x256": dict(shape=(2, 32, 256), rank=6, solver="mu", num_iters=5, num_grad_steps=None, dist="uniform"),
    "hals_r5_16x64": dict(shape=(3, 16, 64), rank=5, solver="hals", num_iters=5, num_grad_steps=None, dist="uniform"),
    "mu_r8_32x128_k3": dict(shape=(2, 2, 32, 128), rank=8, solver="mu", num_iters=5, num_grad_steps=3, dist="uniform"),
}

# --- SWMatricize / Matricize forward + inverse (bit-exact) ---------------------------------------
# name -> dict(input_size, kwargs for ft.SWMatricize, cls)
SW_CASES = {
    # README.md:43-51 geometry at a small spatial size
    "sw3d_hd8_ps8": dict(x_shape=(2, 16, 16, 16, 16), cls="SWMatricize", kw=dict(head_dim=8, patch_size=8)),
    # model_zoo/factorizer_isles22/configs/train.yaml:49-53
    "sw3d_hd8_ps4_s4": dict(x_shape=(1, 8, 8, 8, 8), cls="SWMatricize", kw=dict(head_dim=8, patch_size=4, shifts=[None, 1, 2, 3])),
    # model_zoo/factorizer_brats23/configs/train.yaml:50-54
    "sw3d_hd8_ps8_s4": dict(x_shape=(1, 8, 16, 16, 16), cls="SWMatricize", kw=dict(head_dim=8, patch_size=8, shifts=[None, 2, 4, 6])),
    "sw3d_s3_mixed": dict(x_shape=(1, 4, 8, 12, 16), cls="SWMatricize", kw=dict(num_heads=2, patch_size=(4, 6, 8), shifts=[None, (1, 2, 3), 5])),
    # tests/test_factorizer.py:123
    "sw3d_nh8_ps4": dict(x_shape=(3, 32, 8, 8, 8), cls="SWMatricize", kw=dict(num_heads=8, patch_size=4)),
    "sw2d": dict(x_shape=(2, 8, 16, 24), cls="SWMatricize", kw=dict(num_heads=2, patch_size=(4, 8), shifts=[None, 1, (2, 3)])),
    "sw1d": dict(x_shape=(2, 6, 40), cls="SWMatricize", kw=dict(head_dim=3, patch_size=8)),
    # factorizer/factorizer.py:17 default reshape
    "global3d": dict(x_shape=(2, 16, 8, 8, 8), cls="Matricize", kw=dict(num_heads=1, grid_size=1)),
    "mat3d_shift": dict(x_shape=(1, 8, 8, 8, 16), cls="Matricize", kw=dict(head_dim=4, grid_size=(2, 2, 4), shifts=3)),
}

# --- FactMixer core: reshape -> ReLU -> NMF -> inverse (factorizer/factorizer.py:41-50) ----------
FUSED_CASES = {
    # BASELINE config 2 geometry at 16^3
    "fused_cfg2_16": dict(x_shape=(1, 16, 16, 16, 16), cls="SWMatricize", kw=dict(head_dim=8, patch_size=8),
                          nmf=dict(rank=1, num_iters=5, solver="hals"), relu=True, dist="randn"),
    "fused_cfg2_24_b2": dict(x_shape=(2, 8, 24, 16, 32), cls="SWMatricize", kw=dict(head_dim=8, patch_size=8),
                             nmf=dict(rank=1, num_iters=5, solver="hals"), relu=True, dist="randn"),
    "fused_isles_s4": dict(x_shape=(2, 8, 8, 8, 8), cls="SWMatricize", kw=dict(head_dim=8, patch_size=4, shifts=[None, 1, 2, 3]),
                           nmf=dict(rank=1, num_iters=5, solver="hals"), relu=True, dist="randn"),
    "fused_brats_s4": dict(x_shape=(1, 8, 16, 16, 16), cls="SWMatricize", kw=dict(head_dim=8, patch_size=8, shifts=[None, 2, 4, 6]),
                           nmf=dict(rank=1, num_iters=5, solver="hals"), relu=True, dist="randn"),
    "fused_nh8_ps4": dict(x_shape=(2, 32, 8, 8, 8), cls="SWMatricize", kw=dict(num_heads=8, patch_size=4),
                          nmf=dict(rank=1, num_iters=5, solver="hals"), relu=True, dist="randn"),
    "fused_global_mu": dict(x_shape=(2, 16, 8, 8, 8), cls="Matricize", kw=dict(num_heads=1, grid_size=1),
                            nmf=dict(rank=1, num_iters=5, solver="mu"), relu=True, dist="uniform"),
    # reference default reshape (factorizer/factorizer.py:17, tests/test_factorizer.py:14-110) at sizes beyond one CTA:
    # one grid-wide pass per sweep (csrc/fz_nmf_big.cu)
    "fused_global_mu_big": dict(x_shape=(2, 16, 8, 16, 16), cls="Matricize", kw=dict(num_heads=1, grid_size=1),
                                nmf=dict(rank=1, num_iters=5, solver="mu"), relu=True, dist="uniform"),
    "fused_global_hals_big": dict(x_shape=(1, 32, 8, 8, 24), cls="Matricize", kw=dict(num_heads=1, grid_size=1),
                                  nmf=dict(rank=1, num_iters=5, solver="hals"), relu=True, dist="randn"),
    "fused_global_mu_k2": dict(x_shape=(1, 16, 16, 12, 24), cls="Matricize", kw=dict(num_heads=2, grid_size=1),
                               nmf=dict(rank=1, num_iters=4, solver="mu", num_grad_steps=2), relu=False, dist="uniform"),
    "fused_mu_r2": dict(x_shape=(1, 16, 8, 8, 8), cls="SWMatricize", kw=dict(head_dim=8, patch_size=4),
                        nmf=dict(rank=2, num_iters=5, solver="mu"), relu=False, dist="uniform"),
    "fused_2d": dict(x_shape=(2, 16, 32, 32), cls="SWMatricize", kw=dict(head_dim=4, patch_size=8),
                     nmf=dict(rank=1, num_iters=5, solver="hals"), relu=True, dist="randn"),
    "fused_k2": dict(x_shape=(1, 8, 16, 16, 16), cls="SWMatricize", kw=dict(head_dim=8, patch_size=8),
                     nmf=dict(rank=1, num_iters=5, solver="hals", num_grad_steps=2), relu=True, dist="randn"),
}

# --- FactorizerBlock (factorizer/factorizer.py:60-77), BASELINE config 3 at a small spatial size --
BLOCK_CASES = {
    "block_c16_16": dict(channels=16, spatial=(16, 16, 16), batch=2, mlp_ratio=2,
                         kw=dict(head_dim=8, patch_size=8), nmf=dict(rank=1, num_iters=5, init="uniform", solver="hals")),
    # 32 channels: the fully fused block path (csrc/fz_block_glue.cu); the second one has 384 voxels per
    # sample (a partial 512-voxel tile) and 8x64 windows (generic core kernels)
    "block_c32_16": dict(channels=32, spatial=(16, 16, 16), batch=1, mlp_ratio=2,
                         kw=dict(head_dim=8, patch_size=8), nmf=dict(rank=1, num_iters=5, init="uniform", solver="hals")),
    # mlp_ratio 4 as in model_zoo/factorizer_brats23/configs/train.yaml: hidden width 128 = two slices of the MLP backward
    "block_c32_r4": dict(channels=32, spatial=(8, 8, 8), batch=2, mlp_ratio=4,
                         kw=dict(head_dim=8, patch_size=8), nmf=dict(rank=1, num_iters=5, init="uniform", solver="hals")),
    "block_c32_p4": dict(channels=32, spatial=(4, 8, 12), batch=2, mlp_ratio=1.5,
                         kw=dict(head_dim=8, patch_size=4), nmf=dict(rank=1, num_iters=5, init="uniform", solver="hals")),
    # a width the 32-channel glue kernels do not take, ragged everywhere: 24 channels (not a multiple of the channel map's K chunk),
    # hidden width 36, 320 voxels per sample (2.5 voxel tiles), two samples: _ops.FactorizerBlockWideFn
    "block_c24_p4": dict(channels=24, spatial=(4, 4, 20), batch=2, mlp_ratio=1.5,
                         kw=dict(head_dim=8, patch_size=4), nmf=dict(rank=1, num_iters=5, init="uniform", solver="hals")),
}


# --- whole Swin Factorizer (factorizer/factorizer.py:125-171), README.md:78-96 at a small size --------
MODEL_CASES = {
    # two encoder levels (32 and 64 channels: fused block path and layer-by-layer path), bottleneck with the
    # positional embedding, one decoder level with its 64 -> 32 adapter; eval mode (dropout 0.1 inactive)
    "swin_2level_16": dict(in_channels=2, out_channels=3, spatial=(16, 16, 16), batch=1,
                           kw=dict(encoder_depth=(1, 1), encoder_width=(32, 64), strides=(1, 2), decoder_depth=(1,),
                                   rank=1, num_iters=5, init="uniform", solver="hals", mlp_ratio=2, dropout=0.1),
                           reshape_kw=dict(head_dim=8, patch_size=8)),
}


def _seed(name: str) -> int:
    return int.from_bytes(hashlib.sha256(name.encode()).digest()[:4], "little")


def make_array(name: str, shape, dist: str, tag: str = "x") -> np.ndarray:
    """Deterministic float32 input for case ``name``."""
    rng = np.random.Generator(np.random.PCG64(_seed(name + ":" + tag)))
    if dist == "uniform":
        a = rng.random(shape, dtype=np.float32)
    elif dist == "randn":
        a = rng.standard_normal(shape, dtype=np.float32)
    elif dist == "relu_randn":
        a = np.maximum(rng.standard_normal(shape, dtype=np.float32), 0)
    elif dist == "zero_first":
        a = rng.random(shape, dtype=np.float32)
        a[0] = 0
    else:
        raise ValueError(dist)
    return np.ascontiguousarray(a, dtype=np.float32)


def digest(a: np.ndarray) -> str:
    a = np.ascontiguousarray(a)
    return hashlib.sha256(a.tobytes()).hexdigest()


# --- storage of the golden outputs --------------------------------------------------------------------------------
# Each family (nmf, sw, fused, block, model) is one file, <family>.npz, below 1 MB.  Inputs (u0, v0, state dicts), factors
# and parameter gradients are stored whole.  The outputs y, gx, y64, gx64 of a case with more than SAMPLE[family] entries
# are stored at SAMPLE[family] flat indices drawn once per case from a seeded generator: "<case>/sample_index" and
# "<case>/sample_shape" hold the indices and the full shape, "<key>@sample" the values there.  load_golden returns such
# an output as a Sample, and conftest.tol_ratio compares a computed array with it at those indices.
OUTPUTS = ("y", "gx", "y64", "gx64")
SAMPLE = {"nmf": 1536, "fused": 4096, "block": 8192}


class Sample(np.ndarray):
    """Reference values at the flat indices ``index`` of an array of shape ``full_shape``."""

    def __new__(cls, values, index, full_shape):
        obj = np.asarray(values).view(cls)
        obj.index, obj.full_shape = index, tuple(int(n) for n in full_shape)
        return obj

    def __array_finalize__(self, obj):
        self.index = getattr(obj, "index", None)
        self.full_shape = getattr(obj, "full_shape", None)


def save_golden(directory: str, family: str, arrays: dict) -> None:
    """Write ``arrays`` (insertion order kept) as <directory>/<family>.npz, the larger outputs sampled as above."""
    keep = SAMPLE.get(family)
    out = {}
    for key, a in arrays.items():
        a = np.asarray(a)
        case, name = key.split("/", 1)
        if keep is None or name not in OUTPUTS or a.size <= keep:
            out[key] = a
            continue
        if f"{case}/sample_index" not in out:
            rng = np.random.Generator(np.random.PCG64(_seed(case + ":sample")))
            out[f"{case}/sample_index"] = np.sort(rng.choice(a.size, keep, replace=False)).astype(np.int32)
            out[f"{case}/sample_shape"] = np.array(a.shape, dtype=np.int64)
        assert tuple(out[f"{case}/sample_shape"]) == a.shape, key      # one index set per case
        out[f"{key}@sample"] = a.reshape(-1)[out[f"{case}/sample_index"]]
    path = os.path.join(directory, f"{family}.npz")
    np.savez(path, **out)
    assert os.path.getsize(path) < 1_000_000, (path, os.path.getsize(path))


def load_golden(directory: str, family: str) -> dict:
    """All arrays of ``family`` by key, in the order they were saved; sampled outputs as Sample."""
    with np.load(os.path.join(directory, f"{family}.npz")) as f:
        raw = {k: f[k] for k in f.files}
    out = {}
    for key, a in raw.items():
        if key.endswith("@sample"):
            key = key[:-len("@sample")]
            case = key.split("/", 1)[0]
            out[key] = Sample(a, raw[f"{case}/sample_index"], raw[f"{case}/sample_shape"])
        elif not key.endswith(("/sample_index", "/sample_shape")):
            out[key] = a
    return out
