"""FactorizerBlock forward + backward on bf16 activations against the fp32 block and today's layer-by-layer bf16 autocast route.

Per shape and route, the block step (forward, backward of <out, gout>) is captured in one CUDA graph and replayed; CUDA
events time --reps replays after --warmup.  Routes:
    fp32        x fp32, no autocast: the fused fp32 block (FactorizerBlockFn at 32 channels, FactorizerBlockWideFn otherwise)
    bf16-old    x bf16 under bf16 autocast with the bf16 block path switched off: the layers one by one
    bf16-new    x bf16: FactorizerBlockBf16Fn
The whole Swin Factorizer's training step (forward, sigmoid-BCE + soft-Dice, backward; no optimizer) at 128^3 is timed
eagerly for fp32, bf16-old and bf16-new.  Achieved bandwidth is against the block's algorithmic bytes: every activation
each step reads or writes once, 32 C + 8 H elements per voxel for forward + backward (C channels, H hidden), 4 bytes each
in fp32, 2 in bf16.  Writes JSON (the card's name and power limit included) to --out.

--shifts bundle, --mlp-ratio 4 --batch 2 configure blocks and model like the BraTS23 bundle (shifts [None, 2, 4, 6]).  At
those shifts the fused core took bf16 volumes only after the paired path learnt bf16, so bf16-old also switches the bf16
core off there (FactMixer casts the core's input to fp32, as it did before).  --core adds the core alone at
(--batch, 32, 128^3), fp32 against bf16 on the same path, forward and backward, each as one CUDA graph.

--shifts isles22 configures the ISLES22 bundle's geometry instead: patch 4 (8 x 64 windows on the sub-warp kernels) at shifts
[None, 1, 2, 3], blocks at the stages of a 64^3 ROI, the model at 64^3, the core at (--batch, 32, 64^3); use it with --batch 8.
The fused core took bf16 volumes at patch 4 only after the sub-warp kernels learnt bf16, so bf16-old switches it off there too.

    python bench_probes/bf16_block_time.py --out /tmp/bf16_block_time.json
    python bench_probes/bf16_block_time.py --shifts bundle --mlp-ratio 4 --batch 2 --core --out /tmp/bundle.json
    python bench_probes/bf16_block_time.py --shifts isles22 --batch 8 --core --out /tmp/isles22.json

--dtype f16 times fp16 activations instead (FactorizerBlockF16Fn, fp16 autocast: torch.autocast("cuda")'s default).  Its
routes are fp32, f16-old (fp16 autocast layer by layer with the core cast to fp32, the only fp16 route before the fp16
kernels) and f16-new; the model is timed for fp32, bf16-new (bf16 autocast) and f16-new (fp16 autocast), and --core
compares fp32 with fp16.

    python bench_probes/bf16_block_time.py --dtype f16 --core --out /tmp/f16_block_time.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch
from torch import nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import factorizer_b200 as ft  # noqa: E402
from factorizer_b200 import _ops  # noqa: E402

SHAPES = [(32, 128), (64, 64), (128, 32), (256, 16)]
SHIFTS = {"default": None, "bundle": [None, 2, 4, 6], "isles22": [None, 1, 2, 3]}
DTYPES = {"bf16": torch.bfloat16, "f16": torch.float16}
ISLES22_SHAPES = [(32, 64), (64, 32), (128, 16), (256, 8), (512, 4)]      # (channels, n) of the stages of a 64^3 ROI


def patch_of(shifts):
    return 4 if shifts == SHIFTS["isles22"] else 8


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        return q.stdout.strip().splitlines()[torch.cuda.current_device()]
    except Exception as e:  # noqa: BLE001
        return f"{torch.cuda.get_device_name()} (power limit not read: {e})"


def route_dtype(route):
    return torch.float32 if route == "fp32" else DTYPES[route.split("-")[0]]


class _Route:
    """`route` = fp32, or <bf16|f16>-<old|new>; -old runs under that dtype's autocast with its block path switched off (and its
    core: at the bundle / isles22 shifts for bf16, always for fp16), -new feeds the block that dtype"""
    def __init__(self, name, shifts=None):
        self.name, self.tag = name, name.split("-")[0]
        self.old = name.endswith("-old")
        self.core_off = self.old and (shifts is not None or self.tag == "f16")
        self.saved = (_ops.bf16_block_supported, _ops.bf16_core_supported, _ops.f16_block_supported, _ops.f16_core_supported)

    def __enter__(self):
        if self.old:
            setattr(_ops, f"{self.tag}_block_supported", lambda x, hidden: False)
        if self.core_off:
            setattr(_ops, f"{self.tag}_core_supported", lambda *a, **k: False)
        self.ac = torch.autocast("cuda", dtype=route_dtype(self.name), enabled=self.old)
        self.ac.__enter__()

    def __exit__(self, *exc):
        self.ac.__exit__(*exc)
        _ops.bf16_block_supported, _ops.bf16_core_supported, _ops.f16_block_supported, _ops.f16_core_supported = self.saved


def reshape(shifts):
    kw = {"head_dim": 8, "patch_size": patch_of(shifts)}
    if shifts is not None:
        kw["shifts"] = shifts
    return (ft.SWMatricize, kw)


def block(C, n, ratio=2, shifts=None):
    torch.manual_seed(0)
    return ft.FactorizerBlock(channels=C, spatial_size=(n, n, n), norm=ft.LayerNorm, reshape=reshape(shifts), act=nn.ReLU,
                              factorize=ft.NMF, rank=1, num_iters=5, init="uniform", solver="hals", mlp_ratio=ratio,
                              dropout=0.0).cuda()


def time_graph(fn, warmup, reps):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    for _ in range(warmup):
        g.replay()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def block_leg(B, C, n, route, warmup, reps, ratio=2, shifts=None):
    blk = block(C, n, ratio, shifts)
    H = blk.mlp.block[0].linear.out_channels
    dtype = route_dtype(route)
    x = torch.randn(B, C, n, n, n, device="cuda").to(dtype).requires_grad_(True)
    gout = torch.randn(B, C, n, n, n, device="cuda").to(dtype)
    params = list(blk.parameters())

    def step():
        for p in params:
            p.grad = None
        x.grad = None
        with _Route(route, shifts):
            out = blk(x)
        out.backward(gout.to(out.dtype))
        return out

    with _Route(route, shifts):
        node = type(blk(x).grad_fn).__name__
    ms = time_graph(step, warmup, reps)
    nbytes = (32 * C + 8 * H) * B * n ** 3 * (4 if route == "fp32" else 2)
    del blk
    return {"shape": [B, C, n, n, n], "route": route, "node": node, "ms": ms, "algorithmic_bytes": nbytes,
            "achieved_GBps": nbytes / ms / 1e6}


def model_leg(route, warmup, reps, n=128, B=1, ratio=2, shifts=None):
    torch.manual_seed(1234)
    net = ft.Factorizer(in_channels=4, out_channels=3, spatial_size=(n, n, n), encoder_depth=(1, 1, 1, 1, 1),
                        encoder_width=(32, 64, 128, 256, 512), strides=(1, 2, 2, 2, 2), decoder_depth=(1, 1, 1, 1),
                        norm=ft.LayerNorm, reshape=reshape(shifts), act=nn.ReLU, factorize=ft.NMF, rank=1, num_iters=5,
                        init="uniform", solver="hals", mlp_ratio=ratio, dropout=0.1).cuda()
    net.train()
    x = torch.rand(B, 4, n, n, n, device="cuda")
    target = torch.randint(0, 2, (B, 3, n, n, n), device="cuda").float()

    def step():
        net.zero_grad(set_to_none=True)
        with _Route(route, shifts), torch.autocast("cuda", dtype=route_dtype(route), enabled=route != "fp32"):
            logits = net(x).float()
        p = torch.sigmoid(logits)
        dice = 1 - (2 * (p * target).sum((2, 3, 4)) + 1e-5) / (p.sum((2, 3, 4)) + target.sum((2, 3, 4)) + 1e-5)
        loss = nn.functional.binary_cross_entropy_with_logits(logits, target) + dice.mean()
        loss.backward()

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        step()
    b.record()
    torch.cuda.synchronize()
    return {"route": route, "train_step_ms_eager": a.elapsed_time(b) / reps}


def core_leg(B, shifts, dtype, warmup, reps, C=32, n=128):
    """the fused core alone (SWMatricize -> ReLU -> HALS -> inverse), forward and backward as separate graphs"""
    from factorizer_b200 import _lib
    geom = reshape(shifts)[0]((None, C, n, n, n), **reshape(shifts)[1])._geom
    nmf = ft.NMF((8, patch_of(shifts) ** 3), rank=1, num_iters=5, init="uniform", solver="hals").cuda()
    spec, u0, v0 = nmf.solver_spec(), nmf.init.u0, nmf.init.v0
    x = torch.randn(B, C, n, n, n, device="cuda").to(dtype)
    gy = torch.randn(B, C, n, n, n, device="cuda").to(dtype)
    _, saved = _ops._swnmf_forward(x, u0, v0, geom, spec, True, True)
    path = _lib.lib().fz_last_path()
    fwd = time_graph(lambda: _ops._swnmf_forward(x, u0, v0, geom, spec, True, True), warmup, reps)
    bwd = time_graph(lambda: _ops._swnmf_backward(x, gy, u0, v0, saved, geom, spec, True), warmup, reps)
    return {"shape": [B, C, n, n, n], "dtype": str(dtype), "path": path, "fwd_ms": fwd, "bwd_ms": bwd}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--no-model", action="store_true")
    ap.add_argument("--shifts", choices=sorted(SHIFTS), default="default")
    ap.add_argument("--mlp-ratio", type=int, default=2)
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--core", action="store_true", help="also time the core alone, fp32 against --dtype")
    ap.add_argument("--dtype", choices=sorted(DTYPES), default="bf16", help="the 16-bit activation type of the -old / -new routes")
    args = ap.parse_args()
    old, new = f"{args.dtype}-old", f"{args.dtype}-new"
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    shifts, B = SHIFTS[args.shifts], args.batch
    isles = args.shifts == "isles22"
    n_model = 64 if isles else 128
    res = {"card": card(), "dtype": args.dtype, "shifts": args.shifts, "mlp_ratio": args.mlp_ratio, "batch": B, "core": [], "blocks": [], "model": []}
    if args.core:
        for dtype in (torch.float32, DTYPES[args.dtype]):
            res["core"].append(core_leg(B, shifts, dtype, args.warmup, args.reps, n=n_model))
            print(json.dumps(res["core"][-1]), flush=True)
    for C, n in ISLES22_SHAPES if isles else SHAPES:
        row = {r: block_leg(B, C, n, r, args.warmup, args.reps, args.mlp_ratio, shifts) for r in ("fp32", old, new)}
        row["new_vs_old"] = row[old]["ms"] / row[new]["ms"]
        row["new_vs_fp32"] = row["fp32"]["ms"] / row[new]["ms"]
        res["blocks"].append(row)
        print(json.dumps(row), flush=True)
    if not args.no_model:
        for r in ("fp32", "bf16-old", "bf16-new") if args.dtype == "bf16" else ("fp32", "bf16-new", "f16-new"):
            res["model"].append(model_leg(r, 3, 5, n=n_model, B=B, ratio=args.mlp_ratio, shifts=shifts))
            print(json.dumps(res["model"][-1]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
