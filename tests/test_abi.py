"""The C-ABI library: it loads, exports exactly what include/cdfgpu.h declares, and refuses to work without a GPU
(no CPU fallback).  No compute calls here -- this file runs on the CPU-only build container."""
import re
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def _declared():
    txt = (ROOT / "include" / "cdfgpu.h").read_text()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return set(re.findall(r"\b(cdf(?:gpu|moc|mocsig|zonal|mhst|transig|sigtrp)_\w+)\s*\(", txt))


def test_library_builds_and_exports_every_declared_symbol():
    from cdftools_b200 import build, lib
    so = build.build()
    assert so.exists()
    L = lib.load()
    declared = _declared()
    assert declared, "no prototypes parsed from include/cdfgpu.h"
    for name in declared:
        assert hasattr(L, name), f"{name} declared in cdfgpu.h but not exported by libcdfgpu.so"
    assert declared == set(lib.SIGNATURES), declared ^ set(lib.SIGNATURES)
    assert L.cdfgpu_abi_version() == 1


def test_sass_is_sm100a_only():
    import subprocess
    from cdftools_b200 import build
    out = subprocess.run(["cuobjdump", "-lelf", str(build.build())], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


_NO_DEVICE = """
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from cdftools_b200 import lib
try:
    lib.init(0, 3)
    sys.exit("cdfgpu_init succeeded without a device")
except lib.CdfGpuError as e:
    assert e.code == 5, e.code  # CDFGPU_ERR_NODEVICE
try:
    lib.cdfmoc_submit(0, 0, np.zeros(4, np.float32))
    sys.exit("cdfmoc_gpu_submit succeeded without a device")
except lib.CdfGpuError:
    pass
"""


def test_no_cpu_fallback_without_device():
    """In a process that sees no device (CUDA_VISIBLE_DEVICES empty, so this runs on GPU machines too)."""
    import os
    import subprocess
    import sys
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE, str(ROOT)], capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stdout + r.stderr


def test_product_never_imports_the_oracle():
    for p in (ROOT / "cdftools_b200").rglob("*"):
        if p.suffix in (".py", ".cu", ".cuh", ".inc", ".cpp", ".h", ".f90"):
            txt = p.read_text(errors="ignore")
            assert "import oracle" not in txt and "from oracle" not in txt and "cdf_oracle" not in txt \
                and "libcdforacle" not in txt, p


def test_fortran_module_binds_the_host_facing_abi():
    """cdftools_b200/fortran/cdfgpu_mod.f90 (shipped as source: no Fortran compiler here) names every entry point of
    include/cdfgpu.h that a Fortran host can use; the exceptions take DEVICE pointers or are C-string helpers."""
    fortran = (ROOT / "cdftools_b200" / "fortran" / "cdfgpu_mod.f90").read_text()
    bound = set(re.findall(r"NAME='(\w+)'", fortran))
    device_side_or_c_only = {"cdfmoc_gpu_compute_device", "cdfmoc_gpu_compute_device_batch", "cdfmocsig_gpu_compute_device", "cdfmocsig_gpu_bins_device",
                             "cdfmocsig_gpu_bins_device_stats", "cdfgpu_set_device_inputs_ready", "cdfgpu_microbench", "cdfgpu_h2d_probe",
                             "cdfgpu_strerror", "cdfgpu_launch_count"}
    declared = _declared()
    assert bound <= declared, bound - declared
    assert declared - bound == device_side_or_c_only, (declared - bound) ^ device_side_or_c_only
    # every BIND(C) name is the function's own name (a typo there would only show at link time)
    for fn, name in re.findall(r"FUNCTION\s+(\w+)\s*\([^)]*\)\s*(?:&\s*\n\s*&\s*)?BIND\(C,\s*NAME='(\w+)'\)", fortran):
        assert fn == name, (fn, name)
