"""In-tree nvcc build of the C-ABI library (sm_100a only).  Used by __graft_entry__.build()."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_C")
LIB_PATH = os.path.join(OUT_DIR, "libfactorizer_b200.so")
SOURCES = ["fz_api.cu", "fz_swmat.cu", "fz_nmf_generic.cu", "fz_swnmf_fast.cu", "fz_swnmf_phase.cu", "fz_swnmf_pipe.cu", "fz_layernorm.cu",
           "fz_block_glue.cu", "fz_swnmf_small.cu", "fz_nmf_big.cu", "fz_block_glue_bwd_tc.cu", "fz_block_glue_fwd_tc.cu", "fz_block_glue_lin_tc.cu", "fz_linear.cu", "fz_linear_tc.cu", "fz_bf16_block.cu"]

OBJ_DIR = os.path.join(OUT_DIR, "obj")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
]
LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC", "-cudart", "static"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; factorizer_b200 needs the CUDA 12.9 toolkit to build")


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "factorizer_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def _compile_one(src: str, obj: str, verbose: bool) -> str:
    cmd = [_nvcc(), *NVCC_FLAGS, "-c", "-o", obj, src]
    if os.environ.get("FZ_TUNING"):          # experiment builds (bench_probes/): environment knobs compiled in
        cmd.insert(1, "-DFZ_TUNING")
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed on {src}:\n" + res.stdout + res.stderr)
    return res.stderr


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu into factorizer_b200/_C/libfactorizer_b200.so: one object per source (only the
    stale ones, in parallel), then one link."""
    if not force and not _stale():
        return LIB_PATH
    from concurrent.futures import ThreadPoolExecutor

    obj_dir = OBJ_DIR + ("_tuning" if os.environ.get("FZ_TUNING") else "")      # objects of the two flavours never mix
    os.makedirs(obj_dir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "factorizer_b200.h"))
    headers.append(os.path.abspath(__file__))
    t_hdr = max(os.path.getmtime(h) for h in headers)
    jobs = []
    for s in SOURCES:
        src, obj = os.path.join(CSRC, s), os.path.join(obj_dir, s[:-3] + ".o")
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), t_hdr):
            jobs.append((src, obj))
    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as ex:
        logs = list(ex.map(lambda j: _compile_one(j[0], j[1], verbose), jobs))
    if verbose:
        print("\n".join(logs))
    objs = [os.path.join(obj_dir, s[:-3] + ".o") for s in SOURCES]
    res = subprocess.run([_nvcc(), *LINK_FLAGS, "-o", LIB_PATH, *objs], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
