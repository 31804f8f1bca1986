"""Builds libvp8gpu.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

Each source is compiled to an object under build/ (in parallel, rebuilt only when it or a header changed), then linked.
`build_library(defines=[...], tag="x")` makes a variant library libvp8gpu_x.so for kernel A/B runs (VP8_GPU_LIB selects
it at run time); the product is the untagged one.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
LIB = HERE / "libvp8gpu.so"
SOURCES = [CSRC / "vp8_pairs.cu", CSRC / "vp8_rgb.cu", CSRC / "vp8_png.cu", CSRC / "vp8_pngz.cu", CSRC / "vp8_gpu.cu", CSRC / "vp8_enc.cu", CSRC / "vp8_parse.cpp",
           CSRC / "vp8_alpha.cu", CSRC / "webp_alpha.cpp"]
HEADERS = sorted(list(CSRC.glob("*.h")) + list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.inc")) + list((HERE.parent / "include").glob("*.h")))
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: libvp8gpu.so cannot be built (there is no CPU fallback)")


def _newest_header() -> float:
    return max((p.stat().st_mtime for p in HEADERS if p.exists()), default=0.0)


def stale(lib: Path = LIB) -> bool:
    if not lib.exists():
        return True
    t = lib.stat().st_mtime
    return any(p.exists() and p.stat().st_mtime > t for p in SOURCES + HEADERS)


def build_library(force: bool = False, verbose: bool = False, defines=(), tag: str = "") -> Path:
    lib = HERE / (f"libvp8gpu_{tag}.so" if tag else "libvp8gpu.so")
    if not force and not stale(lib):
        return lib
    nvcc = nvcc_path()
    key = hashlib.sha1((" ".join(defines) + ("|v" if verbose else "")).encode()).hexdigest()[:8]
    objdir = HERE / "build" / (tag or "default")
    objdir.mkdir(parents=True, exist_ok=True)
    hdr_t = _newest_header()

    def compile_one(src: Path) -> Path:
        obj = objdir / f"{src.stem}.{key}.o"
        if not force and obj.exists() and obj.stat().st_mtime > max(src.stat().st_mtime, hdr_t):
            return obj
        cmd = [nvcc, *ARCH, "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC,-O3,-pthread", *[f"-D{d}" for d in defines],
               "-c", "-o", str(obj), str(src)]
        if verbose and src.suffix == ".cu":
            cmd.insert(1, "-Xptxas=-v")
        subprocess.run(cmd, check=True, cwd=str(HERE))
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, [s for s in SOURCES if s.exists()]))
    subprocess.run([nvcc, *ARCH, "-shared", "-o", str(lib), *[str(o) for o in objs]], check=True, cwd=str(HERE))
    # batch CLI front end, linked against the library it sits next to
    cli = CSRC / "vp8gpu_batch.cpp"
    if cli.exists() and not tag:
        subprocess.run(["g++", "-O2", "-std=c++17", "-pthread", "-o", str(HERE / "vp8gpu_batch"), str(cli), "-L" + str(HERE), "-lvp8gpu",
                        "-Wl,-rpath,$ORIGIN"], check=True, cwd=str(HERE))
    return lib


if __name__ == "__main__":
    import sys
    print(build_library(force=True, verbose="-v" in sys.argv))
