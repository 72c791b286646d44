"""Builds ``sygnals_b200/libsygb200.so`` in-tree with nvcc for sm_100a (run: ``python -m sygnals_b200.build``)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libsygb200.so")
SOURCES = [os.path.join(CSRC, f) for f in ("syg_api.cu", "syg_launch_block.cu", "syg_launch_warp.cu", "syg_launch_warp_stft.cu", "syg_launch_stft_ring.cu", "syg_launch_stft_big.cu",
                                             "syg_launch_warp_extra.cu", "syg_launch_warp_spec44k.cu", "syg_launch_warp_spec44kl.cu", "syg_launch_warp_spec22k.cu", "syg_launch_welch.cu", "syg_launch_ingest.cu", "syg_launch_agg.cu", "syg_launch_timefeat.cu", "syg_launch_matrix.cu", "syg_launch_mixed.cu", "syg_launch_warp_res.cu",
                                             "syg_launch_ragged.cu", "syg_launch_ragged_spec.cu")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]
OBJDIR = os.path.join(ROOT, "build", "obj")


def _deps():
    d = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "include", "sygb200.h")]
    return [p for p in d if os.path.isfile(p)]


def up_to_date() -> bool:
    if not os.path.exists(OUT):
        return False
    t = os.path.getmtime(OUT)
    return all(os.path.getmtime(p) <= t for p in _deps())


def build_library(force: bool = False, verbose: bool = False, defines=(), out: str = OUT) -> str:
    """``defines``/``out``: experiment builds (A/B variants of a kernel) into a separate object directory and library file."""
    objdir = OBJDIR if out == OUT else OBJDIR + "_" + os.path.basename(out)
    if not force and out == OUT and up_to_date():
        return OUT
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: libsygb200.so cannot be built (there is no CPU fallback)")
    os.makedirs(objdir, exist_ok=True)
    from concurrent.futures import ThreadPoolExecutor
    hdr_t = max(os.path.getmtime(p) for p in _deps() if not p.endswith(".cu"))

    def compile_one(src):
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= max(hdr_t, os.path.getmtime(src)):
            return obj, ""
        cmd = [nvcc] + NVCC_FLAGS + ["-D" + d for d in defines] + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n" + r.stdout + r.stderr)
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    if verbose:
        for _, log in results:
            sys.stderr.write(log)
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", out + ".tmp"] + [o for o, _ in results]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc link failed:\n" + r.stdout + r.stderr)
    os.replace(out + ".tmp", out)
    return out


if __name__ == "__main__":
    defs = [a[2:] for a in sys.argv[1:] if a.startswith("-D")]
    outs = [a[6:] for a in sys.argv[1:] if a.startswith("--out=")]
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv, defines=defs, out=os.path.abspath(outs[0]) if outs else OUT))
