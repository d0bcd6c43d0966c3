#!/usr/bin/env python
"""Benchmark of the Factorizer hot path on B200 (see BASELINE.json: metric / configs).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload): BASELINE config 3 -- ft.FactorizerBlock(32, 128^3, LayerNorm, SWMatricize(head_dim 8, patch 8),
HALS rank 1 x 5 sweeps, mlp_ratio 2, dropout 0), forward + backward including every parameter gradient, one (1,32,128^3)
fp32 volume per GPU.  A "step" is one forward + one backward through the public module API (ft.FactorizerBlock + autograd).

value      voxels/s with inputs resident in HBM (CUDA events on the launching stream, max over ranks).  The K steps are timed
           as plain stream launches from autograd AND replayed from one CUDA graph per step; the shorter total is reported
           (config.launch says which).
e2e        the same step with HOST buffers: pinned-host x and dOut copied in, out and dX copied out, every step (the copies
           of neighbouring steps overlap the kernels on two side streams)
roofline   the dominant kernel of the step, timed alone over the step's own buffers through its C entry point:
           algorithmic bytes / launch duration against the measured HBM peak (MEASURED_PEAKS.json); `kernels_us` carries
           every kernel group of the step timed the same way
core       BASELINE config 2 (the fused SWMatricize+ReLU+NMF+inverse op inside the block) on its own: forward / backward
           us and the fraction of the HBM roofline of its 20*C bytes per voxel
parity_checked
           max error / tolerance (rtol 1e-4, atol 1e-5) of the TIMED buffers against the oracle, after the timing: the core's
           y and dx against oracle/nmf_oracle.c, the block's out and dx against oracle/block_reference.py
model      configs 4-5: the README Swin Factorizer, inference pass and training step (each also as ONE CUDA graph); under
           torchrun the graphed training step carries the NCCL gradient all-reduce (factorizer_b200/distributed.py: 4 MB
           buckets launched from post-accumulate hooks under the backward), `eager` is the same step under torch
           DistributedDataParallel, and the all-reduce is timed alone too
cpu_baseline / --impl reference
           oracle/torch_port.py -- the reference's PyTorch eager path restated in plain torch (the reference itself is
           pure Python and absent on the GPU box) -- on the SAME workload (the whole block at (1,32,128^3), all host
           threads); the C/OpenMP port of the core (oracle/nmf_oracle.c) is reported beside it
Multi-GPU: one process per GPU (torchrun), batch-sharded (one volume per rank, no data-path collective), weak scaling.

--dump-outputs DIR
           after the timed steps, rank 0 writes what the last timed block step returned to its caller: DIR/out.npy,
           DIR/dx.npy and DIR/grad.<parameter name>.npy, float32.  Inputs and parameters are seeded, so two builds run with
           the same arguments can be compared file by file.  out and dx (2^26 entries each at 128^3) are written as their
           entries at a fixed sample of flat indices (see dump_outputs), about 32 MB in all.  The parameter gradients are
           fp32 sums over 2^21 voxels reduced in no fixed order, so expect them to differ in the last bits from run to
           run; compare them with a tolerance.
--steps K  the number of timed steps of the headline block step (and of --impl reference); the side measurements
           (kernels_us, e2e, model, cpu_baseline) use their own fixed or capped counts.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C, N, HEAD_DIM, PATCH, T_ITERS, HIDDEN = 32, 128, 8, 8, 5, 64
METRIC = "FactorizerBlock voxels/s fwd+bwd @128^3, % of HBM roofline"
UNIT = "voxels/s"
WORKLOAD = ("FactorizerBlock(32,128^3,LayerNorm,SWMatricize(head_dim=8,patch=8,shifts=[None,4]),ReLU,NMF(rank=1,iters=5,hals),"
            "mlp_ratio=2,dropout=0) fwd+bwd incl. parameter gradients on (1,32,128,128,128) fp32 per GPU")
CORE_WORKLOAD = ("SWMatricize(head_dim=8,patch=8,shifts=[None,4])+ReLU+NMF(rank=1,iters=5,hals)+inverse fwd+bwd on "
                 "(1,32,128,128,128) fp32 per GPU (BASELINE config 2)")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------------------------
# CPU arms
# ------------------------------------------------------------------------------------------------------------------
def _host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def torch_port_block(steps: int, warmup: int, budget_s: float | None):
    """The reference's PyTorch CPU path (restated: oracle/torch_port.py) on the whole workload; returns
    (voxels/s, per-step seconds, threads, steps timed).  With a budget, timing stops early once at least two steps
    are timed and the budget is spent."""
    import torch

    from oracle import torch_port as TP

    threads = _host_threads()
    torch.set_num_threads(threads)
    torch.manual_seed(1234)
    import factorizer_b200 as ft      # only for the module's parameter shapes / init (CPU tensors, no kernel runs)
    blk = ft.FactorizerBlock(channels=C, spatial_size=(N, N, N), norm=ft.LayerNorm,
                             reshape=(ft.SWMatricize, {"head_dim": HEAD_DIM, "patch_size": PATCH}),
                             act=torch.nn.ReLU, factorize=ft.NMF, rank=1, num_iters=T_ITERS, init="uniform",
                             solver="hals", mlp_ratio=2, dropout=0.0)
    sd = {k: v.detach().clone().requires_grad_(not k.endswith(("u0", "v0"))) for k, v in blk.state_dict().items()}
    x = torch.rand(1, C, N, N, N, requires_grad=True)
    gy = torch.randn(1, C, N, N, N)
    times, t_start = [], time.perf_counter()
    for k in range(warmup + steps):
        t0 = time.perf_counter()
        y = TP.block_forward(x, sd, HEAD_DIM, (PATCH,) * 3, ((0, 0, 0), (PATCH // 2,) * 3), T_ITERS)
        y.backward(gy)
        x.grad = None
        for v in sd.values():
            v.grad = None
        dt = time.perf_counter() - t0
        if k >= warmup:
            times.append(dt)
        if budget_s is not None and len(times) >= 2 and time.perf_counter() - t_start > budget_s:
            break
    return N ** 3 / statistics.mean(times), times, torch.get_num_threads(), len(times)


def c_port_core(reps: int = 3):
    """oracle/nmf_oracle.c (C/OpenMP restatement of the fused core, config 2) on the whole (1,32,128^3) volume."""
    import numpy as np

    from oracle import c_oracle

    c_oracle.use_all_cores()
    rng = np.random.default_rng(0)
    x = rng.random((1, C, N, N, N), dtype=np.float32)
    gy = rng.standard_normal(x.shape, dtype=np.float32)
    v0 = rng.random(512, dtype=np.float32)
    shifts = [(0, 0, 0), (PATCH // 2,) * 3]
    times = []
    for _ in range(reps + 1):
        t0 = time.perf_counter()
        c_oracle.swnmf_forward(x, v0, HEAD_DIM, (PATCH,) * 3, shifts, relu=True, num_iters=T_ITERS)
        c_oracle.swnmf_backward(x, gy, v0, HEAD_DIM, (PATCH,) * 3, shifts, relu=True, num_iters=T_ITERS)
        times.append(time.perf_counter() - t0)
    times = times[1:]
    return N ** 3 / statistics.median(times), times, c_oracle.num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rate, times, threads, timed = torch_port_block(args.steps, min(args.warmup, 1), budget_s=None)
    sample = (f"the whole workload: FactorizerBlock fwd+bwd on (1,{C},{N}^3), {timed} timed steps "
              f"({statistics.mean(times):.2f} s per step), after {min(args.warmup, 1)} warm-up")
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * statistics.mean(times), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "reference_arm": "oracle/torch_port.py: the reference's PyTorch eager CPU path restated in plain "
                   "torch (same ATen operator sequence, torch autograd); the reference package itself is absent on the GPU box"},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "torch-port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# helpers of the GPU arm
# ------------------------------------------------------------------------------------------------------------------
def bind_to_gpu_cpus(index: int):
    """Run this rank on the CPU cores NVML reports as local to its GPU, so that the pinned host buffers of the
    end-to-end leg are first-touched on the NUMA node next to the GPU.  Returns a short description."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        masks = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(masks) for b in range(64) if (m >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus = cpus & allowed
        if cpus and cpus != allowed:
            os.sched_setaffinity(0, cpus)
            return f"bound to {len(cpus)} GPU-local cores"
        return "all cores are GPU-local"
    except Exception as e:       # no NVML / not permitted: keep the inherited affinity
        return f"not bound ({type(e).__name__})"


class ClockSampler:
    def __init__(self, index: int):
        self.path = f"/tmp/fz_clocks_{os.getpid()}.csv"
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}",
                 "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in open(self.path):
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def tol_ratio(got, ref, rtol=1e-4, atol=1e-5):
    """max |got - ref| / (atol + rtol |ref|) over torch tensors on one device; parity holds when <= 1."""
    import torch
    ref = ref.to(torch.float64)
    return float(((got.to(torch.float64) - ref).abs() / (atol + rtol * ref.abs())).max())


DUMP_SAMPLE = 1 << 22


def dump_outputs(directory, arrays):
    """Write every tensor of `arrays` as <directory>/<name>.npy in float32.  A tensor of more than DUMP_SAMPLE entries is
    reduced to its flattened entries at DUMP_SAMPLE indices drawn by numpy's default_rng(0) (sorted, repeats dropped):
    the same positions in every run."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), DUMP_SAMPLE))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(directory, f"{name}.npy"), t.float().cpu().numpy())


def model_leg(dev, world, rank, n=128, steps=3):
    """Configs 4 and 5 (SURVEY 8d): the README Swin Factorizer on this package's kernels, one 128^3 volume per GPU -- an
    inference pass and a training step (forward, sigmoid-BCE + soft-Dice, backward, AdamW), fp32.  Under torchrun the
    training step runs under DistributedDataParallel over NCCL (gradient all-reduce in 4 MB buckets so that it overlaps the
    backward; model_zoo/factorizer_brats23/configs/train_multigpu.yaml:3-6), and the all-reduce of the same buckets is
    also timed alone.  Side measurement; never raises."""
    import torch
    import torch.distributed as dist
    import factorizer_b200 as ft
    from torch import nn
    keep = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    try:
        torch.backends.cudnn.benchmark = True       # the heuristic choice for the 4->32 stem's fp32 wgrad is 10x slower
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.manual_seed(1234)                      # same initial weights on every rank (DDP broadcasts rank 0's anyway)
        net = ft.Factorizer(in_channels=4, out_channels=3, spatial_size=(n, n, n), encoder_depth=(1, 1, 1, 1, 1),
                            encoder_width=(32, 64, 128, 256, 512), strides=(1, 2, 2, 2, 2), decoder_depth=(1, 1, 1, 1),
                            norm=ft.LayerNorm, reshape=(ft.SWMatricize, {"head_dim": HEAD_DIM, "patch_size": PATCH}),
                            act=nn.ReLU, factorize=ft.NMF, rank=1, num_iters=T_ITERS, init="uniform", solver="hals",
                            mlp_ratio=2, dropout=0.1).to(dev)
        torch.manual_seed(1234 + rank)
        x = torch.rand(1, 4, n, n, n, device=dev)
        target = torch.randint(0, 2, (1, 3, n, n, n), device=dev).float()
        ev = lambda: torch.cuda.Event(enable_timing=True)

        def timed(fn, reps=steps):
            for _ in range(2):
                fn()
            torch.cuda.synchronize(dev)
            if world > 1:
                dist.barrier()
            a, b = ev(), ev()
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            torch.cuda.synchronize(dev)
            return a.elapsed_time(b) / reps

        net.eval()
        with torch.no_grad():
            infer_ms = timed(lambda: net(x))
        net.train()
        params = [q for q in net.parameters() if q.requires_grad]
        nparams = sum(q.numel() for q in params)
        graph_ms = graph_infer_ms = graph_note = None
        red = None
        if True:
            # the same step replayed from ONE CUDA graph (forward, loss, backward, AdamW): the deep stages of the model are
            # launch-bound (a 16^3 or 8^3 stage is a few microseconds of work per kernel), a graph removes the host from them
            try:
                side = torch.cuda.Stream(dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                gopt = torch.optim.AdamW(net.parameters(), lr=1e-4, weight_decay=1e-5, capturable=True, fused=True)
                for q in params:
                    q.grad = None
                # N > 1: this package's bucketed gradient all-reduce (factorizer_b200/distributed.py) -- launched from
                # post-accumulate hooks, so it is part of the captured graph and overlaps the backward
                red = ft.distributed.BucketedGradAllReduce(params, bucket_bytes=4 << 20) if world > 1 else None

                def graph_body():
                    if red is not None:
                        red.zero_grad()
                    else:
                        gopt.zero_grad(set_to_none=True)
                    logits = net(x)
                    p = torch.sigmoid(logits)
                    dice = 1 - (2 * (p * target).sum((2, 3, 4)) + 1e-5) / (p.sum((2, 3, 4)) + target.sum((2, 3, 4)) + 1e-5)
                    loss = nn.functional.binary_cross_entropy_with_logits(logits, target) + dice.mean()
                    loss.backward()
                    if red is not None:
                        red.wait()
                    gopt.step()
                    return loss

                with torch.cuda.stream(side):
                    for _ in range(3):
                        graph_body()
                    if red is None:
                        gopt.zero_grad(set_to_none=True)
                    tg = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(tg, stream=side):
                        graph_body()
                    net.eval()
                    with torch.no_grad():
                        for _ in range(2):
                            net(x)
                        ig = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(ig, stream=side):
                            net(x)
                    net.train()
                torch.cuda.current_stream(dev).wait_stream(side)
                graph_ms = timed(tg.replay)
                graph_infer_ms = timed(ig.replay)
                del tg, ig, gopt
                if red is not None:
                    red.remove()
                    red = None
            except Exception as e:
                graph_note = f"graph capture failed: {type(e).__name__}: {str(e)[:160]}"
                torch.cuda.synchronize(dev)
                if red is not None:
                    red.remove()
        for q in params:
            q.grad = None
        ddp = nn.parallel.DistributedDataParallel(net, device_ids=[dev.index], bucket_cap_mb=4,
                                                  gradient_as_bucket_view=True) if world > 1 else net
        opt = torch.optim.AdamW(net.parameters(), lr=1e-4, weight_decay=1e-5, fused=True)

        def train_step():
            opt.zero_grad(set_to_none=True)
            logits = ddp(x)
            p = torch.sigmoid(logits)
            dice = 1 - (2 * (p * target).sum((2, 3, 4)) + 1e-5) / (p.sum((2, 3, 4)) + target.sum((2, 3, 4)) + 1e-5)
            loss = nn.functional.binary_cross_entropy_with_logits(logits, target) + dice.mean()
            loss.backward()
            opt.step()

        train_ms = timed(train_step)
        out = {"workload": f"Swin Factorizer (README 78-96) 4->3 ch, {n}^3, widths (32,64,128,256,512), HALS r1, B=1/GPU, fp32, "
                           "cudnn.benchmark; all nine blocks run as one autograd node each in this library's kernels (32 channels: "
                           "csrc/fz_block_glue*.cu; 64..512: the tcgen05 channel map with fused epilogues, csrc/fz_linear_tc.cu), so do the "
                           "adapters and the patch (down / up) convolutions as channel maps, the stem's forward and every weight gradient; "
                           "the 3-channel head and the stem backward's pad / unfold are library kernels",
               "params": nparams, "infer_ms": infer_ms, "train_step_ms": train_ms}
        if graph_ms is not None:
            out["eager"] = {"infer_ms": infer_ms, "train_step_ms": train_ms}
            out["infer_ms"], out["train_step_ms"] = min(infer_ms, graph_infer_ms), min(train_ms, graph_ms)
            out["launch"] = "one CUDA graph per training step / per inference pass (eager launches in `eager`)"
        elif graph_note:
            out["launch"] = "eager launches (" + graph_note + ")"
        if world > 1:
            # the collective alone: the same gradient bytes in the same 4 MB buckets, nothing to overlap with
            flat = [torch.zeros(min(1 << 20, nparams - o), device=dev) for o in range(0, nparams, 1 << 20)]

            def allreduce_only():
                for t in flat:
                    dist.all_reduce(t)

            out["allreduce_ms_alone"] = timed(allreduce_only, reps=5)
            out["allreduce_bytes"] = 4 * nparams
            out["train_step"] = (f"forward, sigmoid-BCE + soft-Dice, backward with the NCCL all-reduce (average) of {4 * nparams / 1e6:.1f} MB "
                                 f"of gradients in 4 MB buckets launched from post-accumulate hooks (factorizer_b200/distributed.py) "
                                 f"under the rest of the backward, fused AdamW -- all inside one CUDA graph; `eager` = the same step under "
                                 f"torch DistributedDataParallel (bucket_cap_mb=4) with eager launches; world {world}")
        else:
            out["train_step"] = "forward, sigmoid-BCE + soft-Dice, backward, fused AdamW; single rank: no gradient all-reduce"
        del net, ddp, opt, x, target
        torch.cuda.empty_cache()
        return out
    except Exception as e:                              # a side measurement must not cost the bench line
        try:
            torch.cuda.synchronize(dev)
        except Exception:
            pass
        return {"error": f"{type(e).__name__}: {e}"[:300]}
    finally:
        torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = keep


# ------------------------------------------------------------------------------------------------------------------
# the GPU arm
# ------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    import factorizer_b200 as ft
    from factorizer_b200 import _lib, _ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_cpus(local)       # before any pinned allocation: first touch decides the NUMA node
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.lib()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    stream = torch.cuda.current_stream(dev)
    sp = stream.cuda_stream
    warmup = max(args.warmup, 3)
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---------------- the block (config 3): headline ----------------
    torch.manual_seed(1234 + rank)
    blk = ft.FactorizerBlock(channels=C, spatial_size=(N, N, N), norm=ft.LayerNorm,
                             reshape=(ft.SWMatricize, {"head_dim": HEAD_DIM, "patch_size": PATCH}),
                             act=torch.nn.ReLU, factorize=ft.NMF, rank=1, num_iters=T_ITERS, init="uniform",
                             solver="hals", mlp_ratio=2, dropout=0.0).to(dev)
    with torch.no_grad():       # non-trivial affine parameters (the default init has gamma = 1, beta = 0)
        for nm in ("norm1", "norm2"):
            getattr(blk, nm).norm.weight.add_(0.2 * torch.randn(C, device=dev))
            getattr(blk, nm).norm.bias.add_(0.2 * torch.randn(C, device=dev))
    xb = torch.randn(1, C, N, N, N, device=dev, requires_grad=True)
    gyb = torch.randn(1, C, N, N, N, device=dev)
    block_fused = blk._fused_args(xb) is not None
    plist = list(blk.parameters())

    def clear_grads():
        xb.grad = None
        for p_ in plist:
            p_.grad = None

    def block_step():
        clear_grads()
        out = blk(xb)
        out.backward(gyb)
        return out

    for _ in range(warmup):
        block_step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    _ops.LaunchCounter.total = 0
    b0, b1 = ev(), ev()
    barrier()
    b0.record(stream)
    for _ in range(args.steps):
        out_timed = block_step()
    b1.record(stream)
    barrier()
    total_ms = b0.elapsed_time(b1)
    timed_launches = _ops.LaunchCounter.total
    launch_mode = "stream launches from autograd"
    # what was timed (copies: the autograd graph hanging off `out_timed` must be gone before the capture below, or its
    # AccumulateGrad nodes keep running on this stream and invalidate the capture)
    y_block = out_timed.detach().clone()
    gx_block = xb.grad.detach().clone()
    gp_block = {k: p_.grad.detach().clone() for k, p_ in blk.named_parameters()}
    del out_timed
    bgraph = None
    try:        # the same step replayed from one CUDA graph (forward, autograd backward, gradient accumulation)
        clear_grads()
        cap = torch.cuda.Stream(dev)
        cap.wait_stream(stream)
        with torch.cuda.stream(cap):
            for _ in range(2):
                blk(xb).backward(gyb)
            clear_grads()
            bgraph = torch.cuda.CUDAGraph()
            n_before = _ops.LaunchCounter.total
            with torch.cuda.graph(bgraph, stream=cap):
                out_graph = blk(xb)
                out_graph.backward(gyb)
            per_step_launches = _ops.LaunchCounter.total - n_before
        stream.wait_stream(cap)
        for _ in range(3):
            bgraph.replay()
        barrier()
        b0.record(stream)
        for _ in range(args.steps):
            bgraph.replay()
        b1.record(stream)
        barrier()
        gms = b0.elapsed_time(b1)
        if gms < total_ms:
            total_ms, launch_mode = gms, f"one CUDA graph per step ({per_step_launches} kernel nodes of this library)"
            timed_launches = per_step_launches * args.steps
            y_block = out_graph.detach().clone()
            gx_block = xb.grad.detach().clone()
            gp_block = {k: p_.grad.detach().clone() for k, p_ in blk.named_parameters()}
    except Exception as e:
        launch_mode = f"stream launches from autograd (graph capture failed: {type(e).__name__}: {str(e)[:160]})"
        torch.cuda.synchronize(dev)

    # ---------------- the kernels of one block step, one group at a time, over the step's own kind of buffers ----------------
    sw = blk.fact.reshape
    geom, spec = sw._geom, blk.fact.factorize.solver_spec()
    g, s = geom.c_geom(1), spec.c_solver()
    u0, v0 = blk.fact.factorize.init.u0, blk.fact.factorize.init.v0
    saved = torch.empty(lib.fz_swnmf_saved_bytes(ctypes.byref(g), ctypes.byref(s)), dtype=torch.uint8, device=dev)
    ws = torch.zeros(lib.fz_swnmf_workspace_bytes(ctypes.byref(g), ctypes.byref(s)), dtype=torch.uint8, device=dev)
    n1, n2 = blk.norm1.norm, blk.norm2.norm
    fc1, fc2 = blk.mlp.block[0].linear, blk.mlp.block[3].linear
    w_in, w_out, b_out = blk.fact.in_proj.linear.weight, blk.fact.out_proj.linear.weight, blk.fact.out_proj.linear.bias
    vox = N ** 3
    tz, tm, tx1, tout, td1, td2, td3 = (torch.empty_like(gyb) for _ in range(7))
    gw = [torch.empty_like(t) for t in (n2.weight, n2.bias, fc1.weight, fc1.bias, fc2.weight, fc2.bias, w_out, b_out, w_in, n1.weight, n1.bias)]
    P = lambda t: t.data_ptr()
    xd = xb.detach()

    calls = {
        "ln_linear_fwd (norm1 + in_proj)": lambda: lib.fz_ln_linear_forward(P(xd), P(n1.weight), P(n1.bias), P(w_in), P(tz), 1, C, vox, float(n1.eps), sp),
        "core forward (3 launches)": lambda: lib.fz_swnmf_forward(P(tz), P(u0), P(v0), P(tm), P(saved), P(ws), ctypes.byref(g), ctypes.byref(s), 1, sp),
        "mixer_mlp_fwd (out_proj + residual + norm2 + MLP + residual)": lambda: lib.fz_mixer_mlp_forward(
            P(xd), P(tm), P(w_out), P(b_out), P(n2.weight), P(n2.bias), P(fc1.weight), P(fc1.bias), P(fc2.weight), P(fc2.bias),
            P(tx1), P(tout), 1, C, HIDDEN, vox, float(n2.eps), sp),
        "mlp_bwd (MLP + norm2 backward)": lambda: lib.fz_mlp_backward(
            P(tx1), P(gyb), P(n2.weight), P(n2.bias), P(fc1.weight), P(fc1.bias), P(fc2.weight), P(td1), P(gw[0]), P(gw[1]),
            P(gw[2]), P(gw[3]), P(gw[4]), P(gw[5]), 1, C, HIDDEN, vox, float(n2.eps), sp),
        "linear_bwd (out_proj backward)": lambda: lib.fz_linear_backward(
            P(td1), P(tm), None, None, P(w_out), None, P(td2), P(gw[6]), P(gw[7]), None, None, 1, C, vox, 0.0, 0, sp),
        "core backward (3 launches)": lambda: lib.fz_swnmf_backward(P(tz), P(td2), P(u0), P(v0), P(saved), P(td3), P(ws), ctypes.byref(g), ctypes.byref(s), 1, sp),
        "linear_bwd (in_proj + norm1 backward)": lambda: lib.fz_linear_backward(
            P(td3), P(xd), P(n1.weight), P(n1.bias), P(w_in), P(td1), P(td2), P(gw[8]), None, P(gw[9]), P(gw[10]), 1, C, vox, float(n1.eps), 1, sp),
    }
    # algorithmic volume passes (N_el * 4 bytes each) of every group: inputs read once, outputs written once
    passes = {"ln_linear_fwd (norm1 + in_proj)": 2, "core forward (3 launches)": 2,
              "mixer_mlp_fwd (out_proj + residual + norm2 + MLP + residual)": 4, "mlp_bwd (MLP + norm2 backward)": 3,
              "linear_bwd (out_proj backward)": 3, "core backward (3 launches)": 3, "linear_bwd (in_proj + norm1 backward)": 4}
    kernels_us = {}
    reps = max(5, min(args.steps, 20))
    for name, fn in calls.items():       # in step order: every call finds the inputs the previous ones produced
        for _ in range(2):
            _lib.check(fn())
        a, b = ev(), ev()
        a.record(stream)
        for _ in range(reps):
            _lib.check(fn())
        b.record(stream)
        torch.cuda.synchronize(dev)
        kernels_us[name] = 1e3 * a.elapsed_time(b) / reps
    core_fwd_us, core_bwd_us = kernels_us["core forward (3 launches)"], kernels_us["core backward (3 launches)"]
    core_path = lib.fz_last_path()

    # ---------------- the core on its own (config 2), fwd + bwd back to back: buffers = the block's z / dm ----------------
    for _ in range(3):
        _lib.check(calls["core forward (3 launches)"]()); _lib.check(calls["core backward (3 launches)"]())
    barrier()
    c0, c1 = ev(), ev()
    c0.record(stream)
    for _ in range(args.steps):
        _lib.check(calls["core forward (3 launches)"]()); _lib.check(calls["core backward (3 launches)"]())
    c1.record(stream)
    barrier()
    core_ms = c0.elapsed_time(c1) / args.steps
    core_launch = "stream launches through the C ABI"
    try:        # the same fwd + bwd replayed from one CUDA graph (the C ABI is capturable), as for `value`: the shorter one is reported
        cap = torch.cuda.Stream(dev)
        cap.wait_stream(stream)
        cgraph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cgraph, stream=cap):
            csp = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            _lib.check(lib.fz_swnmf_forward(P(tz), P(u0), P(v0), P(tm), P(saved), P(ws), ctypes.byref(g), ctypes.byref(s), 1, csp))
            _lib.check(lib.fz_swnmf_backward(P(tz), P(td2), P(u0), P(v0), P(saved), P(td3), P(ws), ctypes.byref(g), ctypes.byref(s), 1, csp))
        stream.wait_stream(cap)
        for _ in range(3):
            cgraph.replay()
        barrier()
        c0.record(stream)
        for _ in range(args.steps):
            cgraph.replay()
        c1.record(stream)
        barrier()
        cg_ms = c0.elapsed_time(c1) / args.steps
        if cg_ms < core_ms:
            core_ms, core_launch = cg_ms, "one CUDA graph per fwd+bwd step (6 kernel nodes)"
        del cgraph
    except Exception as e:
        core_launch += f" (graph capture failed: {type(e).__name__}: {str(e)[:120]})"
        torch.cuda.synchronize(dev)

    # ---------------- the same core with bf16 activations (an extension: the reference is fp32) ----------------
    core_bf16 = None
    try:
        gh, = (geom.c_geom(1, torch.bfloat16),)
        zb, dmb = tz.bfloat16(), td2.bfloat16()
        mb_, dzb = torch.empty_like(zb), torch.empty_like(zb)
        fwd_h = lambda: lib.fz_swnmf_forward(P(zb), P(u0), P(v0), P(mb_), P(saved), P(ws), ctypes.byref(gh), ctypes.byref(s), 1, sp)
        bwd_h = lambda: lib.fz_swnmf_backward(P(zb), P(dmb), P(u0), P(v0), P(saved), P(dzb), P(ws), ctypes.byref(gh), ctypes.byref(s), 1, sp)
        for _ in range(3):
            _lib.check(fwd_h()); _lib.check(bwd_h())
        torch.cuda.synchronize(dev)
        h0, h1, h2 = ev(), ev(), ev()
        tf = tb = 0.0
        for _ in range(reps):
            h0.record(stream); _lib.check(fwd_h()); h1.record(stream); _lib.check(bwd_h()); h2.record(stream)
            torch.cuda.synchronize(dev)
            tf += h0.elapsed_time(h1); tb += h1.elapsed_time(h2)
        core_bf16 = {"fwd_us": 1e3 * tf / reps, "bwd_us": 1e3 * tb / reps,
                     "note": "x, y, dy, dx as bf16 (10*C bytes per voxel), arithmetic and factors fp32; parity bound rtol 1e-2 / atol 1e-3 "
                             "(tests/test_gpu_fullsize.py::test_core_bf16_activations)"}
        del zb, dmb, mb_, dzb
    except Exception as e:
        core_bf16 = {"error": f"{type(e).__name__}: {e}"[:200]}
        torch.cuda.synchronize(dev)

    # ---------------- end-to-end with host buffers, through ft.FactorizerBlock + autograd ----------------
    # Every step copies its own x and dOut in from pinned host memory and its out and dX back out; the copy-in of step
    # k+1 and the copy-out of step k-1 run on side streams while step k computes (PCIe is full duplex).
    hx = torch.randn(1, C, N, N, N).pin_memory()
    hgy = torch.randn(1, C, N, N, N).pin_memory()
    hy = torch.empty(1, C, N, N, N).pin_memory()
    hgx = torch.empty(1, C, N, N, N).pin_memory()
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    bufs = [dict(x=torch.empty_like(gyb).requires_grad_(True), gy=torch.empty_like(gyb)) for _ in range(2)]
    in_ready = [torch.cuda.Event() for _ in range(2)]
    comp_done = [torch.cuda.Event() for _ in range(2)]
    out_done = [torch.cuda.Event() for _ in range(2)]
    keep_alive = [None, None]

    def e2e_step(k):
        bfr = bufs[k % 2]
        s_in.wait_event(comp_done[k % 2])          # the kernels of step k-2 have consumed these input buffers
        with torch.cuda.stream(s_in):
            bfr["x"].detach().copy_(hx, non_blocking=True)
            bfr["gy"].copy_(hgy, non_blocking=True)
            in_ready[k % 2].record(s_in)
        stream.wait_event(in_ready[k % 2])
        stream.wait_event(out_done[k % 2])          # step k-2's results have left (their tensors may be recycled now)
        bfr["x"].grad = None
        for p_ in plist:
            p_.grad = None
        out = blk(bfr["x"])
        out.backward(bfr["gy"])
        comp_done[k % 2].record(stream)
        s_out.wait_event(comp_done[k % 2])
        with torch.cuda.stream(s_out):
            hy.copy_(out.detach(), non_blocking=True)
            hgx.copy_(bfr["x"].grad, non_blocking=True)
            out_done[k % 2].record(s_out)
        keep_alive[k % 2] = (out, bfr["x"].grad)    # allocated on the main stream, read on s_out: held until recycled

    e2e_steps = max(4, min(args.steps, 10))
    for k in range(2):
        e2e_step(k)
    barrier()
    e0, e1 = ev(), ev()
    e0.record(stream)
    s_in.wait_event(e0)
    for k in range(e2e_steps):
        e2e_step(k)
    stream.wait_stream(s_out)
    e1.record(stream)
    barrier()
    e2e_ms = e0.elapsed_time(e1) / e2e_steps
    clocks = sampler.stop() if rank == 0 else None
    del bufs, keep_alive, hx, hgy, hy, hgx

    # ---------------- parity of what was timed (rank 0): core vs the C oracle, block vs torch-fp64 + C oracle ----------------
    parity = None
    if rank == 0 and not args.no_parity:
        try:
            from oracle import c_oracle as CO
            from oracle.block_reference import block_reference
            CO.use_all_cores()
            shifts = [(0, 0, 0), (PATCH // 2,) * 3]
            z_np, dm_np, v0_np = tz.cpu().numpy(), td2.cpu().numpy(), v0.detach().cpu().numpy()
            # the core buffers as the last timed core forward / backward left them: m = core(z), dz = core'(z; dm)
            _lib.check(calls["linear_bwd (out_proj backward)"]())      # td2 = dm again (the last group overwrote it with dX)
            _lib.check(calls["core forward (3 launches)"]()); _lib.check(calls["core backward (3 launches)"]())
            torch.cuda.synchronize(dev)
            dm_np = td2.cpu().numpy()
            y_ref = torch.from_numpy(CO.swnmf_forward(z_np, v0_np, HEAD_DIM, (PATCH,) * 3, shifts)).to(dev)
            gx_ref = torch.from_numpy(CO.swnmf_backward(z_np, dm_np, v0_np, HEAD_DIM, (PATCH,) * 3, shifts)).to(dev)
            parity = {"tolerance": "max |err| / (1e-5 + 1e-4 |ref|), <= 1 passes",
                      "core": {"y": tol_ratio(tm, y_ref), "gx": tol_ratio(td3, gx_ref),
                               "oracle": "oracle/nmf_oracle.c on the timed core buffers (z of the block, dm of its backward)"}}
            del y_ref, gx_ref
            o_ref, dx_ref, _, z_ref = block_reference(blk.state_dict(), xd, gyb, tz)
            parity["block"] = {"out": tol_ratio(y_block, o_ref), "gx": tol_ratio(gx_block, dx_ref), "z": tol_ratio(tz, z_ref),
                               "oracle": "oracle/block_reference.py (torch fp64 glue + C-oracle core) on the timed x / dOut"}
            del o_ref, dx_ref, z_ref
        except Exception as e:
            parity = {"error": f"{type(e).__name__}: {e}"[:300]}
        torch.cuda.empty_cache()

    # ---------------- whole model (configs 4 and 5), every rank its own replica (DDP under torchrun) ----------------
    model = None
    if not args.no_model:
        blk = xb = bgraph = out_graph = None
        del tz, tm, tx1, tout, td1, td2, td3, saved, ws
        torch.cuda.empty_cache()
        model = model_leg(dev, world, rank)
        barrier()

    # ---------------- reduce over ranks ----------------
    dom_name = max(kernels_us, key=lambda k: kernels_us[k])
    vals = torch.tensor([total_ms, e2e_ms, core_ms, core_fwd_us, core_bwd_us, kernels_us[dom_name]], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, core_ms, core_fwd_us, core_bwd_us, dom_us = vals.tolist()
    if model and world > 1 and "train_step_ms" in model:
        mv = torch.tensor([model["train_step_ms"], model["infer_ms"], model.get("allreduce_ms_alone", 0.0)], device=dev, dtype=torch.float64)
        dist.all_reduce(mv, op=dist.ReduceOp.MAX)
        model["train_step_ms"], model["infer_ms"], model["allreduce_ms_alone"] = mv.tolist()

    if rank == 0:
        peak, peak_src = load_peaks()
        n_el = C * N ** 3
        voxels = N ** 3
        ms_per_step = total_ms / args.steps
        floor_bytes = 5 * n_el * 4          # x, dOut in; out, dX out ... = 20*C bytes per voxel (SURVEY 8d)
        dom_bytes = passes[dom_name] * n_el * 4
        achieved = dom_bytes / (dom_us * 1e-6) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                traffic = json.load(f).get(dom_name)
        if model and "train_step_ms" in model:
            model["train_voxels_per_s"] = world * voxels / (model["train_step_ms"] * 1e-3)
            model["infer_voxels_per_s"] = world * voxels / (model["infer_ms"] * 1e-3)
        if core_bf16 and "fwd_us" in core_bf16:
            hb = 1e-3 * (core_bf16["fwd_us"] + core_bf16["bwd_us"])
            core_bf16["ms_per_step"] = hb
            core_bf16["voxels_per_s_per_gpu"] = voxels / (hb * 1e-3)
            core_bf16["hbm_frac_of_its_own_bytes"] = (floor_bytes / 2) / (hb * 1e-3) / 1e9 / peak
            core_bf16["speedup_vs_fp32_core"] = core_ms / hb
        line = {
            "metric": METRIC, "value": world * voxels / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "volumes_per_gpu": 1, "parallelism": f"batch-sharded x{world}, no data-path collective",
                       "l2": "inputs and saved activations (6 x 256 MiB per step) are larger than the 126 MB L2; no explicit flush",
                       "host_affinity": numa, "launch": launch_mode,
                       "path": ("fused glue kernels (csrc/fz_block_glue*.cu) around the fused core (csrc/fz_swnmf_phase.cu): 5 launches forward, 6 backward"
                                if block_fused else "layer by layer around the fused core"),
                       "block_hbm_frac_of_absolute_floor": floor_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                       "e2e_scaling_note": "e2e is bound by the host: every rank streams 1 GiB per step through pinned memory of the same "
                                           "host (about 46 GB/s per direction per GPU alone, ~120 GB/s shared), so it does not scale with N"},
            "roofline": {"bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": dom_bytes, "kernel_us": dom_us,
                         "note": "the dominant kernel group of the block step, timed alone through its C entry point; kernels_us lists all "
                                 "of them with their algorithmic volume passes (x N_el x 4 bytes)",
                         "kernels_us": kernels_us, "kernel_passes": passes},
            "core": {"workload": CORE_WORKLOAD, "ms_per_step": core_ms, "voxels_per_s": world * voxels / (core_ms * 1e-3),
                     "fwd_us": core_fwd_us, "bwd_us": core_bwd_us, "launch": core_launch,
                     "fused_op_hbm_frac": floor_bytes / (core_ms * 1e-3) / 1e9 / peak,
                     "path": {0: "generic", 1: "window-at-a-time", 2: "octant kernels, three launches per direction", 6: "octant kernels, one pipelined launch"}.get(core_path, str(core_path))},
            "core_bf16": core_bf16,
            "e2e": {"value": world * voxels / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": 2 * n_el * 4, "d2h_bytes_per_step": 2 * n_el * 4,
                    "api": "ft.FactorizerBlock(...)(x).backward(dOut) on tensors copied from / to pinned host memory every step"},
            "gpu_launches": timed_launches,
            "parity_checked": parity,
            "clocks": clocks,
        }
        if model:
            line["model"] = model
        if world == 1 and not args.no_cpu:
            os.sched_setaffinity(0, all_cpus)       # the CPU baseline gets every core again
            rate, times, threads, timed = torch_port_block(2, 1, budget_s=60.0)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": threads, "kind": "torch-port",
                                    "sample": f"the whole workload: FactorizerBlock fwd+bwd on (1,{C},{N}^3) through oracle/torch_port.py "
                                              f"(the reference's PyTorch eager path restated), 1 warm-up + {timed} timed steps, "
                                              f"{statistics.mean(times):.2f} s per step"}
            crate, ctimes, cthreads = c_port_core(3)
            line["cpu_baseline_c_port"] = {"value": crate, "unit": UNIT, "cores": cthreads, "kind": "port",
                                           "sample": f"the fused core alone (config 2) on the whole (1,{C},{N}^3) volume through "
                                                     f"oracle/nmf_oracle.c (C/OpenMP), median of 3 ({1e3 * statistics.median(ctimes):.0f} ms)"}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"out": y_block, "dx": gx_block, **{f"grad.{k}": g for k, g in gp_block.items()}})
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the headline block step (and of --impl reference)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-model", action="store_true", help="skip the whole-model (configs 4-5) side measurement")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity check of the timed buffers")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output and gradients under DIR (.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
