"""Build recipe of libcdfgpu.so (the C-ABI CUDA library) -- sm_100a only, in-tree, no JIT cache.

    python -m cdftools_b200.build            # builds cdftools_b200/libcdfgpu.so if sources are newer
    python -m cdftools_b200.build --force

nvcc cross-compiles without a GPU.  Flags that matter for parity:
  -fmad=false            no implicit FMA contraction in device code (the reference's gfortran -O build on
                         baseline x86-64 emits none; the sigma-bin assignment must be bit-exact)
  -Xcompiler -ffp-contract=off   same for the host-side reference-profile polynomial
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
SO = PKG / "libcdfgpu.so"
SOURCES = [CSRC / "api.cu"]
DEPS = [CSRC / n for n in ("api.cu", "api_mocsig.inc", "api_zonal.inc", "common.cuh", "moc_kernel.cuh", "mocsig_kernel.cuh", "mocsig_filter.hpp", "eos_device.cuh", "microbench.cuh", "moc_decomp.cuh",
                            "zonal_kernels.cuh", "transig_kernels.cuh", "api_transig.inc", "api_multi.inc", "unpack_kernels.cuh")] + [
    PKG.parent / "include" / "cdfgpu.h", PKG.parent / "include" / "cdf_eos_coeffs.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17", "-fmad=false",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-O2",
    "-Xptxas", "-v",
    "-shared", "-cudart", "static",
]


def nvcc_path() -> str:
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and Path(c).exists():
            return c
    raise RuntimeError("nvcc not found: libcdfgpu.so cannot be built (there is no CPU fallback)")


def needs_build() -> bool:
    if not SO.exists():
        return True
    t = SO.stat().st_mtime
    return any(d.stat().st_mtime > t for d in DEPS)


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not needs_build():
        return SO
    cmd = [nvcc_path(), *NVCC_FLAGS, "-ccbin", "/usr/bin/g++" if Path("/usr/bin/g++").exists() else "g++",
           "-o", str(SO), *map(str, SOURCES)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    log = r.stdout + r.stderr
    (PKG / "build.log").write_text(" ".join(cmd) + "\n" + log)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + log[-4000:])
    if verbose:
        print(log)
    return SO


HOST = CSRC / "host"
HOST_TOOLS = {"cdfmoc_gpu": "cdfmoc_main.cpp", "cdfmocsig_gpu": "cdfmocsig_main.cpp", "cdfmhst_gpu": "cdfmhst_main.cpp",
              "cdfzonalsum_gpu": "cdfzonal_main.cpp", "cdfzonalmean_gpu": "cdfzonal_main.cpp",
              "cdftransig_xy3d_gpu": "cdftransig_main.cpp", "cdfsigtrp_gpu": "cdfsigtrp_main.cpp", "nc3dump": "nc3dump_main.cpp"}
HOST_DEFINES = {"cdfzonalmean_gpu": ["-DZONAL_MEAN"]}


def build_host(force: bool = False, bindir: Path | None = None, names=None) -> dict:
    """C++ twins of the cdfmoc / cdfmocsig command lines (NetCDF-3 I/O + the C ABI) into bindir (default cdftools_b200/bin/):
    the tools named in `names`, every tool by default."""
    build(force=False)
    bindir = Path(bindir) if bindir is not None else PKG / "bin"
    bindir.mkdir(parents=True, exist_ok=True)
    out = {}
    cxx = "/usr/bin/g++" if Path("/usr/bin/g++").exists() else "g++"
    hdrs = [HOST / "nc3.hpp", HOST / "host_common.hpp", PKG.parent / "include" / "cdfgpu.h"]
    for name in names or HOST_TOOLS:
        src = HOST_TOOLS[name]
        exe = bindir / name
        deps = [HOST / src] + hdrs + ([SO] if name != "nc3dump" else [])
        if force or not exe.exists() or any(d.stat().st_mtime > exe.stat().st_mtime for d in deps):
            cmd = [cxx, "-O2", "-std=c++17", "-Wall", "-pthread", "-ffp-contract=off", *HOST_DEFINES.get(name, []), "-o", str(exe), str(HOST / src)]
            if name != "nc3dump":
                cmd += ["-L" + str(PKG), "-lcdfgpu", "-Wl,-rpath," + str(PKG), "-Wl,-rpath,$ORIGIN/.."]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("g++ failed for %s:\n%s" % (name, (r.stdout + r.stderr)[-4000:]))
        out[name] = exe
    return out


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose=True)
    print("built", p)
    print("built", ", ".join(str(v) for v in build_host(force="--force" in sys.argv).values()))
