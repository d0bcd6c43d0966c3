"""The Swin Factorizer's scaffold layers (stem, strided down-samplers, transposed up-samplers, decoder adapters, 1x1 head) under
bf16 autocast: this library's bf16 kernels (_ops.bf16_layer_supported) against the library route (cuDNN / cuBLAS, reached by
switching the predicate off).

Per layer of the README model at 128^3 and route, forward + backward of <y, g> is captured in one CUDA graph and replayed; CUDA
events time --reps replays after --warmup.  Inputs are what the model hands each layer: the stem gets the fp32 volume, the
first up-sampler the bottleneck's fp32 output, every other layer bf16.  Then the model's training step (forward, sigmoid-BCE +
soft-Dice, backward; no optimizer): fp32, and bf16 autocast with the library scaffold, with this library's kernels on every
scaffold layer, and with the predicate as shipped (the library where it measured faster), each eager and from a CUDA graph.  Writes JSON (the card's name and power limit included) to --out.

    python bench_probes/bf16_scaffold_time.py --out /tmp/bf16_scaffold_time.json
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
from factorizer_b200 import _ops, layers  # noqa: E402

N = 128
# name: (module factory, input shape, input dtype)
LAYERS = {
    "stem 4->32 @128^3": (lambda: layers.Conv3d(4, 32, kernel_size=3, padding=1, bias=False), (1, 4, N, N, N), torch.float32),
    "down 32->64 @128^3": (lambda: layers.Conv3d(32, 64, kernel_size=2, stride=2), (1, 32, N, N, N), torch.bfloat16),
    "down 64->128 @64^3": (lambda: layers.Conv3d(64, 128, kernel_size=2, stride=2), (1, 64, 64, 64, 64), torch.bfloat16),
    "down 128->256 @32^3": (lambda: layers.Conv3d(128, 256, kernel_size=2, stride=2), (1, 128, 32, 32, 32), torch.bfloat16),
    "down 256->512 @16^3": (lambda: layers.Conv3d(256, 512, kernel_size=2, stride=2), (1, 256, 16, 16, 16), torch.bfloat16),
    "up 512->256 @8^3": (lambda: layers.ConvTranspose3d(512, 256, kernel_size=2, stride=2), (1, 512, 8, 8, 8), torch.float32),
    "up 256->128 @16^3": (lambda: layers.ConvTranspose3d(256, 128, kernel_size=2, stride=2), (1, 256, 16, 16, 16), torch.bfloat16),
    "up 128->64 @32^3": (lambda: layers.ConvTranspose3d(128, 64, kernel_size=2, stride=2), (1, 128, 32, 32, 32), torch.bfloat16),
    "up 64->32 @64^3": (lambda: layers.ConvTranspose3d(64, 32, kernel_size=2, stride=2), (1, 64, 64, 64, 64), torch.bfloat16),
    "adapter 512->256 @16^3": (lambda: ft.Linear(512, 256, bias=False), (1, 512, 16, 16, 16), torch.bfloat16),
    "adapter 256->128 @32^3": (lambda: ft.Linear(256, 128, bias=False), (1, 256, 32, 32, 32), torch.bfloat16),
    "adapter 128->64 @64^3": (lambda: ft.Linear(128, 64, bias=False), (1, 128, 64, 64, 64), torch.bfloat16),
    "adapter 64->32 @128^3": (lambda: ft.Linear(64, 32, bias=False), (1, 64, N, N, N), torch.bfloat16),
    "head 32->3 @128^3": (lambda: layers.Conv3d(32, 3, kernel_size=1), (1, 32, N, N, N), torch.bfloat16),
    "bottleneck linear 512->1024 @8^3": (lambda: ft.Linear(512, 1024), (1, 512, 8, 8, 8), torch.float32),
}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        return q.stdout.strip().splitlines()[torch.cuda.current_device()]
    except Exception as e:  # noqa: BLE001
        return f"{torch.cuda.get_device_name()} (power limit not read: {e})"


class _Route:
    """Under bf16 autocast -- library: the scaffold predicate off; new: this library's bf16 kernels on every layer the kernels
    take (_ops.bf16_library_faster off); rule: the predicate as shipped.  fp32: no autocast."""

    def __init__(self, name):
        self.name = name
        self.saved = (_ops.bf16_layer_supported, _ops.bf16_library_faster)

    def __enter__(self):
        if self.name == "library":
            _ops.bf16_layer_supported = lambda *a, **k: False
        if self.name == "new":
            _ops.bf16_library_faster = lambda *a, **k: False
        self.ac = torch.autocast("cuda", dtype=torch.bfloat16, enabled=self.name != "fp32", cache_enabled=False)
        self.ac.__enter__()

    def __exit__(self, *exc):
        self.ac.__exit__(*exc)
        _ops.bf16_layer_supported, _ops.bf16_library_faster = self.saved


def _time(fn, warmup, reps, graph):
    if graph:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                fn()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        fn = g.replay
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def layer_leg(name, route, warmup, reps):
    make, shape, dtype = LAYERS[name]
    torch.manual_seed(0)
    m = make().cuda()
    x = torch.randn(*shape, device="cuda").to(dtype).requires_grad_(not name.startswith("stem"))
    with _Route(route):
        y = m(x)
    g = torch.randn_like(y)
    node = type(y.grad_fn).__name__
    del y                                   # no autograd graph outlives this call: the capture makes its own

    def step():
        for p in m.parameters():
            p.grad = None
        x.grad = None
        with _Route(route):
            out = m(x)
        out.backward(g)

    return {"layer": name, "route": route, "node": node, "ms": _time(step, warmup, reps, graph=True)}


def _node_chain(y, depth=3):
    names, frontier = [], [y.grad_fn]
    for _ in range(depth):
        names += [type(fn).__name__ for fn in frontier if fn is not None]
        frontier = [f for fn in frontier if fn is not None for f, _ in fn.next_functions]
    return names


def model_leg(route, graph, warmup, reps):
    torch.manual_seed(1234)
    net = ft.Factorizer(in_channels=4, out_channels=3, spatial_size=(N, N, N), encoder_depth=(1, 1, 1, 1, 1),
                        encoder_width=(32, 64, 128, 256, 512), strides=(1, 2, 2, 2, 2), decoder_depth=(1, 1, 1, 1),
                        norm=ft.LayerNorm, reshape=(ft.SWMatricize, {"head_dim": 8, "patch_size": 8}), act=nn.ReLU,
                        factorize=ft.NMF, rank=1, num_iters=5, init="uniform", solver="hals", mlp_ratio=2, dropout=0.1).cuda()
    net.train()
    x = torch.rand(1, 4, N, N, N, device="cuda")
    target = torch.randint(0, 2, (1, 3, N, N, N), device="cuda").float()

    def step():
        net.zero_grad(set_to_none=not graph)
        with _Route(route):
            logits = net(x).float()
        p = torch.sigmoid(logits)
        dice = 1 - (2 * (p * target).sum((2, 3, 4)) + 1e-5) / (p.sum((2, 3, 4)) + target.sum((2, 3, 4)) + 1e-5)
        loss = nn.functional.binary_cross_entropy_with_logits(logits, target) + dice.mean()
        loss.backward()

    ms = _time(step, warmup, reps, graph)
    del net
    return {"route": route, "mode": "graph" if graph else "eager", "train_step_ms": ms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--no-model", action="store_true")
    args = ap.parse_args()
    res = {"card": card(), "layers": [], "model": []}
    print(res["card"], flush=True)
    for name in LAYERS:
        row = {r: layer_leg(name, r, args.warmup, args.reps) for r in ("library", "new")}
        row["new_vs_library"] = row["library"]["ms"] / row["new"]["ms"]
        with _Route("rule"):
            make, shape, dtype = LAYERS[name]
            chain = _node_chain(make().cuda()(torch.zeros(*shape, device="cuda", dtype=dtype)))
        row["rule_takes"] = "new" if any("Bf16" in n for n in chain) else "library"
        res["layers"].append(row)
        print(json.dumps(row), flush=True)
    if not args.no_model:
        for graph in (False, True):
            for r in ("fp32", "library", "new", "rule"):
                res["model"].append(model_leg(r, graph, 3, 10))
                print(json.dumps(res["model"][-1]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
