"""Build libmvg_b200.so (sm_100a) in-tree with nvcc.  Used by __graft_entry__.build() and by hand:
    python multiview-clustering_b200/build.py
The shared library lands in multiview-clustering_b200/mvc_b200/ so that it travels with gpurun."""
from __future__ import annotations

import os
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
OUT = HERE / "mvc_b200" / "libmvg_b200.so"
SOURCES = ["mv_capi.cu", "mv_draw_simt.cu", "mv_draw_tc.cu", "mv_state_kernels.cu", "mv_stats_tile.cu", "mv_summary.cu", "mv_counts.cu", "mv_exchange.cu", "mv_seq.cu"]
# per-file overrides: the sequential engine must not contract a*b+c (the compiled reference does not either)
EXTRA = {"mv_seq.cu": ["--fmad=false"]}
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "--fmad=true", "-Xptxas", "-v"]


def needs_build() -> bool:
    if not OUT.exists():
        return True
    t = OUT.stat().st_mtime
    deps = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.h")) + \
        [HERE.parent / "include" / "mvg.h", Path(__file__)]
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not needs_build():
        return OUT
    objdir = HERE / "build"
    objdir.mkdir(exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        obj = objdir / (src + ".o")
        objs.append(str(obj))
        flags = [f for f in FLAGS if not (src in EXTRA and f == "--fmad=true")] + EXTRA.get(src, [])
        cmd = [NVCC, *flags, "-c", str(CSRC / src), "-o", str(obj)]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"== {src}\n{out}")
        if p.returncode != 0:
            sys.stderr.write("\n".join(log))
            raise RuntimeError(f"nvcc failed on {src}")
    (objdir / "ptxas.log").write_text("\n".join(log))
    if verbose:
        print("\n".join(log))
    link = [NVCC, "-shared", "--cudart", "static", "-o", str(OUT), *objs, "-ldl"]
    subprocess.run(link, check=True)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
