"""In-tree build of libes3.so (sm_100a only): `python -m efficientsam3_b200.build`.

nvcc cross-compiles without a GPU.  Each .cu is compiled to an object (parallel, cached by mtime)
and linked into efficientsam3_b200/libes3.so, which is git-ignored but travels to the GPU box.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
OBJ = HERE / "build"
LIB = HERE / "libes3.so"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _needs(src: Path, obj: Path, deps: list[Path]) -> bool:
    if not obj.exists():
        return True
    t = obj.stat().st_mtime
    return any(d.stat().st_mtime > t for d in [src, *deps])


def build(verbose: bool = False, force: bool = False) -> Path:
    OBJ.mkdir(exist_ok=True)
    srcs = sorted(CSRC.glob("*.cu"))
    hdrs = sorted(CSRC.glob("*.cuh"))
    nvcc = _nvcc()
    jobs = []
    for s in srcs:
        o = OBJ / (s.stem + ".o")
        if force or _needs(s, o, hdrs):
            cmd = [nvcc, *NVCC_FLAGS, "-c", str(s), "-o", str(o)]
            if verbose:
                cmd.insert(1, "-Xptxas")
                cmd.insert(2, "-v")
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        if verbose:
            sys.stderr.write(r.stderr)

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        list(ex.map(run, jobs))
    objs = [str(OBJ / (s.stem + ".o")) for s in srcs]
    # relink when an object is newer than the library too: a build stopped between compiling and linking left it stale
    if jobs or force or not LIB.exists() or any(os.path.getmtime(o) > LIB.stat().st_mtime for o in objs):
        tmp = LIB.with_suffix(".so.tmp")     # link beside the target, then rename: a reader never sees a half-written library
        run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(tmp), *objs, "-lcudart"])
        os.replace(tmp, LIB)
    return LIB


if __name__ == "__main__":
    p = build(verbose="-v" in sys.argv, force="-f" in sys.argv)
    print(p)
