"""Build rrtplanner_b200/librrtk.so (hand-written sm_100a CUDA behind the C ABI of include/rrtk.h).

    python -m rrtplanner_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the
repository snapshot; nothing is JIT-compiled at run time.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "librrtk.so")
SOURCES = ["api.cu", "grid.cu", "inflate.cu", "collision.cu", "clearance.cu", "queries.cu", "rng.cu", "plan.cu", "plan_wide.cu",
           "plan_scan_standard.cu", "plan_scan_star.cu", "plan_scan_informed.cu", "plan_grid.cu", "plan_rewire.cu", "peaks.cu",
           "shortcut.cu", "disc.cu", "body.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "--fmad=false",            # cost arithmetic must be mul / add / sqrt in IEEE double, never fused
    "-Xcompiler", "-fPIC", "-Xptxas", "-v",
]


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "rrtk.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, out: str = None, extra=()) -> str:
    """``out`` / ``extra``: experiment builds (other output path, extra nvcc flags such as -D...)."""
    if out is None and not force and not needs_build():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    tag = "" if out is None else "." + os.path.basename(out)
    out = out or OUT
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", tag + ".o"))
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, p in procs:
        text, _ = p.communicate()
        log.append(f"== {src}\n{text}")
        if p.returncode:
            sys.stderr.write("\n".join(log))
            raise RuntimeError(f"nvcc failed on {src}")
    subprocess.check_call([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out, *objs])
    with open(os.path.join(HERE, "build", "ptxas%s.log" % tag), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
