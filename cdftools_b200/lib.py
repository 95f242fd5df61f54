"""ctypes binding of libcdfgpu.so -- every call goes through the C ABI declared in include/cdfgpu.h.

This is the Python twin of the Fortran ISO_C_BINDING module (cdftools_b200/fortran/cdfgpu_mod.f90): same entry
points, same argument meaning.  There is no CPU implementation behind it: if the shared library is missing or no
CUDA device is usable, the calls raise CdfGpuError.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

PKG = Path(__file__).resolve().parent
import os

# CDFGPU_LIB: path of an alternative build of the library (A/B experiments with compile-time variants, tools/ab_variants.sh)
SO_PATH = Path(os.environ["CDFGPU_LIB"]) if os.environ.get("CDFGPU_LIB") else PKG / "libcdfgpu.so"

EOS80, TEOS10, NEUTRAL = 0, 1, 2
INPUT_F32, INPUT_I16 = 0, 1                      # cdfgpu_set_input_packing types
FIELD_ZV, FIELD_ZT, FIELD_ZS, FIELD_ZVEIV, FIELD_E3V_VVL = range(5)   # ... and fields (order of the submit arguments)
CALL_ZONAL, CALL_MHST, CALL_MHST_VTS, CALL_TRANSIG = range(4)         # cdfgpu_set_sibling_input calls

# name -> (restype, argtypes): the complete export list of include/cdfgpu.h (tests check both directions)
_f32p, _f64p, _i16p, _i32p = C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_int16), C.POINTER(C.c_int32)
SIGNATURES = {
    "cdfgpu_init": (C.c_int, [C.c_int, C.c_int]),
    "cdfgpu_init_multi": (C.c_int, [C.c_int, C.c_int, C.c_int]),
    "cdfgpu_warmup": (C.c_int, []),
    "cdfgpu_num_devices": (C.c_int, []),
    "cdfgpu_nslots": (C.c_int, []),
    "cdfgpu_finalize": (C.c_int, []),
    "cdfgpu_synchronize": (C.c_int, []),
    "cdfgpu_strerror": (C.c_char_p, [C.c_int]),
    "cdfgpu_last_error": (C.c_char_p, []),
    "cdfgpu_device_count": (C.c_int, []),
    "cdfgpu_abi_version": (C.c_int, []),
    "cdfgpu_pinned_alloc": (C.c_void_p, [C.c_size_t]),
    "cdfgpu_pinned_free": (C.c_int, [C.c_void_p]),
    "cdfgpu_launch_count": (C.c_ulonglong, []),
    "cdfgpu_h2d_probe": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.POINTER(C.c_double)]),
    "cdfgpu_set_input_big_endian": (C.c_int, [C.c_int]),
    "cdfgpu_set_input_packing": (C.c_int, [C.c_int, C.c_int, C.c_float, C.c_float, C.c_float]),
    "cdfgpu_set_sibling_input": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float]),
    "cdfgpu_set_device_inputs_ready": (C.c_int, [C.c_int]),
    "cdfgpu_microbench": (C.c_int, [C.c_int, C.POINTER(C.c_double)]),
    "cdfmoc_gpu_setup": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cdfmoc_gpu_set_e3v": (C.c_int, [C.c_void_p]),
    "cdfmoc_gpu_submit": (C.c_int, [C.c_int, C.c_int, C.c_void_p]),
    "cdfmoc_gpu_fetch": (C.c_int, [C.c_int, C.c_void_p]),
    "cdfmoc_gpu_compute_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "cdfmoc_gpu_compute_device_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "cdfmoc_gpu_kernel_ms": (C.c_int, [C.c_int, C.POINTER(C.c_float)]),
    "cdfmoc_gpu_maxmoc": (C.c_int, [C.c_int] * 6 + [C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "cdfmoc_gpu_decomp_setup": (C.c_int, [C.c_int] + [C.c_void_p] * 5),
    "cdfmoc_gpu_decomp_submit": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cdfmoc_gpu_decomp_fetch": (C.c_int, [C.c_int] + [C.c_void_p] * 4),
    "cdfmoc_gpu_decomp_device": (C.c_int, [C.c_void_p] * 8),
    "cdfmoc_gpu_maxmoc_windows": (C.c_int, [C.c_int, C.c_void_p]),
    "cdfmoc_gpu_maxmoc_device": (C.c_int, [C.c_void_p] * 4),
    "cdfmoc_gpu_teardown": (C.c_int, []),
    "cdfmocsig_gpu_setup": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float,
                                      C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_float,
                                      C.c_int, C.c_int]),
    "cdfmocsig_gpu_submit": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cdfmocsig_gpu_fetch": (C.c_int, [C.c_int, C.c_void_p]),
    "cdfmocsig_gpu_set_isodep": (C.c_int, [C.c_void_p]),
    "cdfmocsig_gpu_fetch_isodep": (C.c_int, [C.c_int, C.c_void_p]),
    "cdfmocsig_gpu_compute_device": (C.c_int, [C.c_void_p] * 7),
    "cdfmocsig_gpu_compute_device_isodep": (C.c_int, [C.c_void_p] * 8),
    "cdfmocsig_gpu_bins_device": (C.c_int, [C.c_void_p] * 4),
    "cdfmocsig_gpu_bins_device_stats": (C.c_int, [C.c_void_p] * 3 + [C.POINTER(C.c_ulonglong), C.c_void_p]),
    "cdfmocsig_gpu_filter_info": (C.c_int, [C.POINTER(C.c_double)]),
    "cdfmocsig_gpu_kernel_ms": (C.c_int, [C.c_int, C.POINTER(C.c_float)]),
    "cdfmocsig_gpu_teardown": (C.c_int, []),
    "cdfzonal_gpu_setup": (C.c_int, [C.c_int] * 4 + [C.c_void_p] * 4),
    "cdfzonal_gpu_sum": (C.c_int, [C.c_void_p] * 3),
    "cdfzonal_gpu_mean": (C.c_int, [C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cdfzonal_gpu_submit_sum": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p]),
    "cdfzonal_gpu_submit_mean": (C.c_int, [C.c_int, C.c_void_p, C.c_float, C.c_int]),
    "cdfzonal_gpu_fetch": (C.c_int, [C.c_int] + [C.c_void_p] * 3),
    "cdfzonal_gpu_kernel_ms": (C.c_int, [C.POINTER(C.c_float)]),
    "cdfzonal_gpu_teardown": (C.c_int, []),
    "cdfzonal_gpu_sum_device": (C.c_int, [C.c_void_p] * 4),
    "cdfzonal_gpu_mean_device": (C.c_int, [C.c_void_p, C.c_float, C.c_int] + [C.c_void_p] * 4),
    "cdfmhst_gpu_setup": (C.c_int, [C.c_int] * 3 + [C.c_void_p] * 6),
    "cdfmhst_gpu_record": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "cdfmhst_gpu_record_vts": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "cdfmhst_gpu_submit": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "cdfmhst_gpu_submit_vts": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "cdfmhst_gpu_fetch": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p]),
    "cdfmhst_gpu_kernel_ms": (C.c_int, [C.POINTER(C.c_float)]),
    "cdfmhst_gpu_teardown": (C.c_int, []),
    "cdfmhst_gpu_record_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 3),
    "cdfmhst_gpu_record_vts_device": (C.c_int, [C.c_void_p] * 3 + [C.c_int] + [C.c_void_p] * 3),
    "cdftransig_gpu_setup": (C.c_int, [C.c_int] * 4 + [C.c_float, C.c_int, C.c_double, C.c_double, C.c_int] + [C.c_void_p] * 5 + [C.c_int]),
    "cdftransig_gpu_record": (C.c_int, [C.c_void_p] * 6 + [C.c_int]),
    "cdftransig_gpu_fetch": (C.c_int, [C.c_void_p, C.c_void_p]),
    "cdftransig_gpu_submit": (C.c_int, [C.c_int] + [C.c_void_p] * 6 + [C.c_int]),
    "cdftransig_gpu_wait": (C.c_int, [C.c_int]),
    "cdftransig_gpu_kernel_ms": (C.c_int, [C.POINTER(C.c_float)]),
    "cdftransig_gpu_teardown": (C.c_int, []),
    "cdftransig_gpu_record_device": (C.c_int, [C.c_void_p] * 6 + [C.c_int, C.c_void_p]),
    "cdftransig_gpu_fetch_device": (C.c_int, [C.c_void_p] * 3),
    "cdfsigtrp_gpu_section": (C.c_int, [C.c_int] * 3 + [C.c_void_p] * 9 + [C.c_int, C.c_float, C.c_int, C.c_double, C.c_double, C.c_int]
                              + [C.c_void_p] * 6),
    "cdfsigtrp_gpu_kernel_ms": (C.c_int, [C.POINTER(C.c_float)]),
    "cdfsigtrp_gpu_sections_setup": (C.c_int, [C.c_int] * 4 + [C.c_void_p] * 10 + [C.c_float] * 3 + [C.c_int, C.c_float, C.c_int, C.c_double,
                                                                                                     C.c_double, C.c_int, C.c_void_p, C.c_void_p]),
    "cdfsigtrp_gpu_sections_device": (C.c_int, [C.c_void_p] * 7),
    "cdfsigtrp_gpu_teardown": (C.c_int, []),
}


class CdfGpuError(RuntimeError):
    def __init__(self, code: int, where: str, text: str):
        super().__init__(f"{where}: error {code}: {text}")
        self.code = code


_lib = None


def load():
    """dlopen libcdfgpu.so and declare all prototypes.  Fails loudly if the library has not been built."""
    global _lib
    if _lib is None:
        if not SO_PATH.exists():
            raise CdfGpuError(-1, "load", f"{SO_PATH} is missing -- build it with `python -m cdftools_b200.build` "
                                          "(there is no CPU fallback)")
        lib = C.CDLL(str(SO_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def _chk(rc: int, where: str):
    if rc != 0:
        lib = load()
        raise CdfGpuError(rc, where, (lib.cdfgpu_last_error() or b"").decode() or lib.cdfgpu_strerror(rc).decode())


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    if isinstance(a, np.ndarray):
        assert a.flags["C_CONTIGUOUS"], "array must be C-contiguous ([k][j][i] == Fortran (i,j,k))"
        return C.c_void_p(a.ctypes.data)
    if hasattr(a, "data_ptr"):  # torch tensor (host pinned or device)
        assert a.is_contiguous()
        return C.c_void_p(a.data_ptr())
    raise TypeError(type(a))


def stream_handle(stream) -> int:
    """cudaStream_t for the C ABI from a torch stream.  torch's default stream is handle 0, which the ABI reserves
    for "the library's own compute stream"; map it to cudaStreamLegacy (0x1)."""
    if stream is None:
        return 0
    h = int(stream.cuda_stream) if hasattr(stream, "cuda_stream") else int(stream)
    return h if h != 0 else 1


# ---- lifecycle -----------------------------------------------------------------------------------------------
_device = 0   # CUDA ordinal of the library's (first) device: where the tensors of the *_device calls must live


def init(device: int = -1, nslots: int = 0):
    global _device
    _chk(load().cdfgpu_init(device, nslots), "cdfgpu_init")
    _device = device if device >= 0 else int(os.environ.get("CDFGPU_DEVICE", "0"))


def init_multi(ndev: int, shard: str = "time", nslots: int = 0):
    """One process, several devices: shard = "time" (slot s on device s mod N) or "lat" (latitude bands)."""
    global _device
    _chk(load().cdfgpu_init_multi(int(ndev), {"time": 0, "lat": 1}[shard], nslots), "cdfgpu_init_multi")
    _device = int(os.environ.get("CDFGPU_DEVICE", "0"))


def num_devices() -> int:
    return int(load().cdfgpu_num_devices())


def nslots() -> int:
    return int(load().cdfgpu_nslots())


def finalize():
    if _lib is not None:
        _chk(_lib.cdfgpu_finalize(), "cdfgpu_finalize")
        _drop()
        _plans.clear()


def synchronize():
    _chk(load().cdfgpu_synchronize(), "cdfgpu_synchronize")


def device_count() -> int:
    return int(load().cdfgpu_device_count())


def launch_count() -> int:
    return int(load().cdfgpu_launch_count())


def set_input_big_endian(on: bool):
    _chk(load().cdfgpu_set_input_big_endian(int(bool(on))), "cdfgpu_set_input_big_endian")


def set_input_packing(field: int, kind: int, scale_factor=1.0, add_offset=0.0, spval=0.0):
    """Field `field` of the submit calls (FIELD_*) is handed over as int16 values (kind INPUT_I16, e.g. an np.int16 array
    or PinnedArray(shape, np.int16)) and unpacked on the device as getvar does, or as float32 (INPUT_F32, the default)."""
    _chk(load().cdfgpu_set_input_packing(int(field), int(kind), float(scale_factor), float(add_offset), float(spval)),
         "cdfgpu_set_input_packing")


def set_sibling_input(call: int, field: int, kind: int, big_endian=False, scale_factor=1.0, add_offset=0.0, spval=0.0):
    """Record array `field` of the sibling call `call` (CALL_*; fields in the order of the call's arguments) is handed over
    as int16 values (kind INPUT_I16, unpacked on the device as getvar does) or float32 (INPUT_F32, the default), in host
    byte order or, with big_endian, as the raw bytes of the file."""
    _chk(load().cdfgpu_set_sibling_input(int(call), int(field), int(kind), int(bool(big_endian)), float(scale_factor),
                                         float(add_offset), float(spval)), "cdfgpu_set_sibling_input")


class PinnedArray:
    """A numpy view over a page-locked buffer from cdfgpu_pinned_alloc (what NF90_GET_VAR would fill)."""

    def __init__(self, shape, dtype=np.float32):
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        self.addr = load().cdfgpu_pinned_alloc(self.nbytes)
        if not self.addr:
            raise CdfGpuError(4, "cdfgpu_pinned_alloc", load().cdfgpu_last_error().decode())
        buf = (C.c_char * self.nbytes).from_address(self.addr)
        self.array = np.frombuffer(buf, dtype=dtype).reshape(shape)

    def free(self):
        if self.addr:
            self.array = None
            load().cdfgpu_pinned_free(self.addr)
            self.addr = None


# ---- cdfmoc ----------------------------------------------------------------------------------------------------
def cdfmoc_setup(e1v, e3v_masked, ibmask):
    """e1v (ny,nx) f32; e3v_masked (nz,ny,nx) f32 already * vmask (cdfmoc.f90:590-594); ibmask (ny,nx,nb) int16."""
    nz, ny, nx = e3v_masked.shape
    nb = ibmask.shape[2]
    assert e1v.shape == (ny, nx) and ibmask.shape[:2] == (ny, nx)
    assert e1v.dtype == np.float32 and e3v_masked.dtype == np.float32 and ibmask.dtype == np.int16
    _plans.pop("moc", None)
    _chk(load().cdfmoc_gpu_setup(nx, ny, nz, nb, _ptr(e1v), _ptr(e3v_masked), _ptr(ibmask)), "cdfmoc_gpu_setup")
    _plans["moc"] = dict(n3=(nz - 1) * ny * nx, nout=nz * ny * nb, nwin=0)
    return (nz, ny, nb)


def cdfmoc_set_e3v(e3v_masked):
    _chk(load().cdfmoc_gpu_set_e3v(_ptr(e3v_masked)), "cdfmoc_gpu_set_e3v")


def cdfmoc_submit(slot: int, jt: int, zv):
    _chk(load().cdfmoc_gpu_submit(slot, jt, _ptr(zv)), "cdfmoc_gpu_submit")


def cdfmoc_fetch(slot: int, out):
    _chk(load().cdfmoc_gpu_fetch(slot, _ptr(out)), "cdfmoc_gpu_fetch")
    return out


def cdfmoc_compute_device(d_zv, d_dmoc, stream=None):
    _chk(load().cdfmoc_gpu_compute_device(_ptr(d_zv), _ptr(d_dmoc), C.c_void_p(stream_handle(stream))),
         "cdfmoc_gpu_compute_device")


def cdfmoc_compute_device_batch(d_zv_list, d_dmoc_list, stream=None):
    """One K1 launch over several device-resident records (lists of torch tensors / device addresses)."""
    n = len(d_zv_list)
    assert n == len(d_dmoc_list) and n >= 1
    addr = lambda a: a.data_ptr() if hasattr(a, "data_ptr") else int(a)
    zv = (C.c_void_p * n)(*[addr(a) for a in d_zv_list])
    out = (C.c_void_p * n)(*[addr(a) for a in d_dmoc_list])
    _chk(load().cdfmoc_gpu_compute_device_batch(zv, out, n, C.c_void_p(stream_handle(stream))), "cdfmoc_gpu_compute_device_batch")


def cdfmoc_kernel_ms(slot: int) -> float:
    ms = C.c_float()
    _chk(load().cdfmoc_gpu_kernel_ms(slot, C.byref(ms)), "cdfmoc_gpu_kernel_ms")
    return ms.value


def cdfmoc_decomp_setup(e1u, gphiv, gdept, umask, tmask, teos10=False):
    """umask, tmask: int16 (>= nz-1, ny, nx) planes as the reference reads them (cdfmoc.f90:439-440)."""
    assert umask.dtype == np.int16 and tmask.dtype == np.int16 and e1u.dtype == np.float32
    gphiv32 = np.ascontiguousarray(gphiv, np.float32)   # held in locals: a converted temporary must outlive the C call
    gdept32 = np.ascontiguousarray(gdept, np.float32)
    _chk(load().cdfmoc_gpu_decomp_setup(int(teos10), _ptr(e1u), _ptr(gphiv32), _ptr(gdept32), _ptr(umask), _ptr(tmask)),
         "cdfmoc_gpu_decomp_setup")


def cdfmoc_decomp_submit(slot, jt, zv, zt, zs):
    _chk(load().cdfmoc_gpu_decomp_submit(slot, jt, _ptr(zv), _ptr(zt), _ptr(zs)), "cdfmoc_gpu_decomp_submit")


def cdfmoc_decomp_fetch(slot, shape):
    outs = {k: np.empty(shape, np.float64) for k in ("total", "sh", "bt", "ag")}
    _chk(load().cdfmoc_gpu_decomp_fetch(slot, _ptr(outs["total"]), _ptr(outs["sh"]), _ptr(outs["bt"]), _ptr(outs["ag"])),
         "cdfmoc_gpu_decomp_fetch")
    return outs


def cdfmoc_decomp_device(d_zv, d_zt, d_zs, d_dmoc, d_dmoc_sh, d_dmoc_bt, d_dmoc_ag, stream=None):
    """-decomp of a device-resident record, enqueued on `stream` (a torch stream or handle; None: the library's): d_zv, d_zt,
    d_zs (nz-1,ny,nx) f32 into the total and the three components, each (nz,ny,nb) f64 -- torch CUDA tensors or device
    addresses."""
    p = _plans.get("moc", {})
    fields = [_dev(a, name, p.get("n3"), "float32") for name, a in (("d_zv", d_zv), ("d_zt", d_zt), ("d_zs", d_zs))]
    outs = [_dev(a, name, p.get("nout"), "float64") for name, a in (("d_dmoc", d_dmoc), ("d_dmoc_sh", d_dmoc_sh),
                                                                      ("d_dmoc_bt", d_dmoc_bt), ("d_dmoc_ag", d_dmoc_ag))]
    _chk(load().cdfmoc_gpu_decomp_device(*fields, *outs, C.c_void_p(stream_handle(stream))), "cdfmoc_gpu_decomp_device")


def cdfmoc_maxmoc_windows(windows):
    """The cdfmaxmoc windows of the following cdfmoc_maxmoc_device calls: a sequence of (basin, ijmin, ijmax, ikmin, ikmax),
    basin 0-based, the window 1-based inclusive as cdfmoc_maxmoc takes them."""
    win = np.ascontiguousarray(np.asarray(windows, np.int32).reshape(-1, 5))
    _chk(load().cdfmoc_gpu_maxmoc_windows(int(win.shape[0]), _ptr(win)), "cdfmoc_gpu_maxmoc_windows")
    if "moc" in _plans:
        _plans["moc"]["nwin"] = int(win.shape[0])


def cdfmoc_maxmoc_device(d_dmoc, d_ovt, d_loc, stream=None):
    """Every window of cdfmoc_maxmoc_windows over the device slab d_dmoc (nz,ny,nb) f64 in one launch: d_ovt (nwin,2) f32 =
    max, min; d_loc (nwin,4) int32 = (jj, jk) of the max, (jj, jk) of the min, 1-based."""
    p = _plans.get("moc", {})
    nwin = p.get("nwin") or None
    _chk(load().cdfmoc_gpu_maxmoc_device(_dev(d_dmoc, "d_dmoc", p.get("nout"), "float64"),
                                         _dev(d_ovt, "d_ovt", nwin and 2 * nwin, "float32"),
                                         _dev(d_loc, "d_loc", nwin and 4 * nwin, "int32"), C.c_void_p(stream_handle(stream))),
         "cdfmoc_gpu_maxmoc_device")


def maxmoc_window(rlat, gdepw, latmin, latmax, depmin, depmax):
    """Index window of cdfmaxmoc (src/cdfmaxmoc.f90:145-155): the LAST index whose latitude / depth is <= the limit.
    rlat (ny,) and gdepw (nz,) as cdfmaxmoc holds them (gdepw = -depthw of the file, positive down).  1-based."""
    ijmin = ijmax = ikmin = ikmax = 0
    for jj, v in enumerate(rlat, 1):
        if v <= latmin: ijmin = jj
        if v <= latmax: ijmax = jj
    for jk, v in enumerate(gdepw, 1):
        if v <= depmin: ikmin = jk
        if v <= depmax: ikmax = jk
    return ijmin, ijmax, ikmin, ikmax


def cdfmoc_maxmoc(slot, basin, ijmin, ijmax, ikmin, ikmax):
    """-> (ovtmax, ovtmin, (jj,jk) of max, (jj,jk) of min), 1-based, on the slot's device slab."""
    ovt = (C.c_float * 2)()
    loc = (C.c_int * 4)()
    _chk(load().cdfmoc_gpu_maxmoc(slot, basin, ijmin, ijmax, ikmin, ikmax, ovt, loc), "cdfmoc_gpu_maxmoc")
    return ovt[0], ovt[1], (loc[0], loc[1]), (loc[2], loc[3])


def cdfmoc_teardown():
    _chk(load().cdfmoc_gpu_teardown(), "cdfmoc_gpu_teardown")
    _plans.pop("moc", None)


# ---- cdfmocsig -------------------------------------------------------------------------------------------------
def cdfmocsig_setup(e1v, e3v, ibmask, nz, nbins, sigmin, sigstp, pref, eos, spv=0.0, spt=0.0, sps=0.0,
                    j_first_global=0, ny_global=None):
    """e3v (>=nz-1,ny,nx) f32 UNmasked, or None with -vvl (then every submit brings e3v)."""
    ny, nx = e1v.shape
    nb = ibmask.shape[2]
    assert e1v.dtype == np.float32 and ibmask.dtype == np.int16 and ibmask.shape[:2] == (ny, nx)
    if e3v is not None:
        assert e3v.dtype == np.float32 and e3v.shape[0] >= nz - 1 and e3v.shape[1:] == (ny, nx)
    _plans.pop("mocsig", None)
    _chk(load().cdfmocsig_gpu_setup(nx, ny, nz, nb, int(nbins), float(sigmin), float(sigstp), float(pref), int(eos),
                                    _ptr(e1v), _ptr(e3v), _ptr(ibmask), float(spv), float(spt), float(sps),
                                    int(j_first_global), int(ny if ny_global is None else ny_global)),
         "cdfmocsig_gpu_setup")
    _plans["mocsig"] = dict(n3=(nz - 1) * ny * nx, nout=ny * int(nbins) * nb)
    return (ny, int(nbins), nb)


def cdfmocsig_submit(slot, jt, zv, zt, zs, zveiv=None, e3v_vvl=None):
    _chk(load().cdfmocsig_gpu_submit(slot, jt, _ptr(zv), _ptr(zt), _ptr(zs), _ptr(zveiv), _ptr(e3v_vvl)),
         "cdfmocsig_gpu_submit")


def cdfmocsig_fetch(slot, out):
    _chk(load().cdfmocsig_gpu_fetch(slot, _ptr(out)), "cdfmocsig_gpu_fetch")
    return out


def cdfmocsig_set_isodep(gdept):
    gdept32 = None if gdept is None else np.ascontiguousarray(gdept, np.float32)   # kept alive across the C call
    _chk(load().cdfmocsig_gpu_set_isodep(_ptr(gdept32)), "cdfmocsig_gpu_set_isodep")


def cdfmocsig_fetch_isodep(slot, out):
    _chk(load().cdfmocsig_gpu_fetch_isodep(slot, _ptr(out)), "cdfmocsig_gpu_fetch_isodep")
    return out


def cdfmocsig_compute_device(d_zv, d_zt, d_zs, d_dmoc, d_zveiv=None, d_e3v_vvl=None, stream=None):
    _chk(load().cdfmocsig_gpu_compute_device(_ptr(d_zv), _ptr(d_zt), _ptr(d_zs), _ptr(d_zveiv), _ptr(d_e3v_vvl),
                                             _ptr(d_dmoc), C.c_void_p(stream_handle(stream))),
         "cdfmocsig_gpu_compute_device")


def cdfmocsig_compute_device_isodep(d_zv, d_zt, d_zs, d_dmoc, d_depi, d_zveiv=None, d_e3v_vvl=None, stream=None):
    """cdfmocsig_compute_device with -isodep (cdfmocsig_set_isodep first): d_zv, d_zt, d_zs, d_zveiv, d_e3v_vvl (nz-1,ny,nx)
    f32 into d_dmoc and d_depi (ny,nbins,nb) f64 -- torch CUDA tensors or device addresses."""
    p = _plans.get("mocsig", {})
    fields = [_dev(a, name, p.get("n3"), "float32") for name, a in (("d_zv", d_zv), ("d_zt", d_zt), ("d_zs", d_zs),
                                                                     ("d_zveiv", d_zveiv), ("d_e3v_vvl", d_e3v_vvl))]
    _chk(load().cdfmocsig_gpu_compute_device_isodep(*fields, _dev(d_dmoc, "d_dmoc", p.get("nout"), "float64"),
                                                    _dev(d_depi, "d_depi", p.get("nout"), "float64"),
                                                    C.c_void_p(stream_handle(stream))),
         "cdfmocsig_gpu_compute_device_isodep")


def set_device_inputs_ready(on: bool = True):
    """Records handed to *_compute_device on a caller stream are resident and synchronised (see cdfgpu.h)."""
    _chk(load().cdfgpu_set_device_inputs_ready(1 if on else 0), "cdfgpu_set_device_inputs_ready")


def h2d_probe(pinned: "PinnedArray", reps: int = 4) -> float:
    """GB/s of plain pinned-host -> device copies on the copy stream (the platform ceiling of *_submit's input leg)."""
    v = C.c_double()
    _chk(load().cdfgpu_h2d_probe(C.c_void_p(pinned.addr), C.c_size_t(pinned.nbytes), int(reps), C.byref(v)), "cdfgpu_h2d_probe")
    return float(v.value)


def microbench() -> dict:
    """Measured issue ceilings: {name: (warp-instructions / clock / SM, Ginst/s over the chip, SM MHz)}."""
    out = {}
    for kind, name in enumerate(("dfma", "ffma", "ffma2", "int", "ffma_int_mix")):
        v = (C.c_double * 3)()
        _chk(load().cdfgpu_microbench(kind, v), "cdfgpu_microbench")
        out[name] = {"winst_per_clk_sm": v[0], "ginst_per_s": v[1], "sm_mhz": v[2]}
    return out


def cdfmocsig_bins_device_stats(d_zt, d_zs, d_ibin, stream=None):
    """Bins of a device-resident record plus (cells, cells past the fp32 tier, cells on the reference chain)."""
    st = (C.c_ulonglong * 3)()
    _chk(load().cdfmocsig_gpu_bins_device_stats(_ptr(d_zt), _ptr(d_zs), _ptr(d_ibin), st, C.c_void_p(stream_handle(stream))),
         "cdfmocsig_gpu_bins_device_stats")
    return int(st[0]), int(st[1]), int(st[2])


def cdfmocsig_filter_info() -> dict:
    v = (C.c_double * 8)()
    _chk(load().cdfmocsig_gpu_filter_info(v), "cdfmocsig_gpu_filter_info")
    return {"tier1": bool(v[0]), "tier2": bool(v[1]), "err32_kgm3": v[2], "margin32_bins": v[3], "margin64_bins": v[4],
            "chunks_per_row": int(v[5]), "levels_per_chunk": int(v[6]), "resident_ctas": int(v[7])}


def cdfmocsig_bins_device(d_zt, d_zs, d_ibin, stream=None):
    _chk(load().cdfmocsig_gpu_bins_device(_ptr(d_zt), _ptr(d_zs), _ptr(d_ibin), C.c_void_p(stream_handle(stream))),
         "cdfmocsig_gpu_bins_device")


def cdfmocsig_kernel_ms(slot: int) -> float:
    ms = C.c_float()
    _chk(load().cdfmocsig_gpu_kernel_ms(slot, C.byref(ms)), "cdfmocsig_gpu_kernel_ms")
    return ms.value


def cdfmocsig_teardown():
    _chk(load().cdfmocsig_gpu_teardown(), "cdfmocsig_gpu_teardown")
    _plans.pop("mocsig", None)


# ---- sibling tools (SURVEY.md section 8 f3) ----------------------------------------------------------------------
def _c32(a):
    a = np.ascontiguousarray(a, np.float32)
    return a


def _rec(a):
    """A record array of a sibling call: int16 (a field declared INPUT_I16 with set_sibling_input) goes as it is, anything
    else as float32."""
    if isinstance(a, np.ndarray) and a.dtype == np.int16:
        return np.ascontiguousarray(a)
    return _c32(a)


# tool -> element counts of its current plan, which the *_device wrappers check tensors against
_plans: dict = {}


def _dev(a, what: str, n, dtype: str):
    """A device array of a *_device call: a torch CUDA tensor of `dtype` ("float32" / "float64"), contiguous, on the library's
    device and of n elements (when the plan is known), or a raw device address (int) passed as it is.  ValueError otherwise:
    a host array would reach the kernels as a device pointer."""
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    if not (hasattr(a, "data_ptr") and getattr(a, "is_cuda", False)):
        raise ValueError(f"{what}: expected a CUDA tensor or a device address, got {type(a).__name__}")
    if str(a.dtype) != "torch." + dtype:
        raise ValueError(f"{what}: dtype {a.dtype}, expected torch.{dtype}")
    if not a.is_contiguous():
        raise ValueError(f"{what}: the tensor is not contiguous")
    if a.device.index != _device:
        raise ValueError(f"{what}: the tensor is on {a.device}, the library on cuda:{_device}")
    if n is not None and a.numel() != n:
        raise ValueError(f"{what}: {a.numel()} elements, the plan has {n}")
    return C.c_void_p(a.data_ptr())


def cdfzonal_setup(e1, e2, zmask, zmaskvar):
    """e1, e2 (ny,nx) f32; zmask (ny,nx,nb) f32 (basin fastest); zmaskvar (nk,ny,nx) f32."""
    e1, e2, zmask, zmaskvar = _c32(e1), _c32(e2), _c32(zmask), _c32(zmaskvar)
    nk, ny, nx = zmaskvar.shape
    nb = zmask.shape[2]
    assert e1.shape == (ny, nx) and e2.shape == (ny, nx) and zmask.shape[:2] == (ny, nx)
    _chk(load().cdfzonal_gpu_setup(nx, ny, nk, nb, _ptr(e1), _ptr(e2), _ptr(zmask), _ptr(zmaskvar)), "cdfzonal_gpu_setup")
    _drop("zonal")
    _plans["zonal"] = dict(n3=nk * ny * nx, ny=ny, nout=nb * nk * ny)
    return nb, nk, ny


def cdfzonal_sum(zv, shape, alpha=None):
    """zv (nk,ny,nx) f32 (or int16, see set_sibling_input) -> dzosum (nb,nk,ny) f64; shape = the tuple cdfzonal_setup returned."""
    zv = _rec(zv)
    out = np.empty(shape, np.float64)
    al = _c32(alpha) if alpha is not None else None
    _chk(load().cdfzonal_gpu_sum(_ptr(zv), _ptr(al), _ptr(out)), "cdfzonal_gpu_sum")
    return out


def cdfzonal_mean(zv, shape, zspval=0.0, lmax=False):
    """-> (dzomean (nb,nk,ny) f64, rzomax, rzomin (nb,nk,ny) f32 or None)."""
    zv = _rec(zv)
    mean = np.empty(shape, np.float64)
    zmax = np.empty(shape, np.float32) if lmax else None
    zmin = np.empty(shape, np.float32) if lmax else None
    _chk(load().cdfzonal_gpu_mean(_ptr(zv), float(zspval), int(lmax), _ptr(mean), _ptr(zmax), _ptr(zmin)), "cdfzonal_gpu_mean")
    return mean, zmax, zmin


def cdfzonal_sum_device(d_zv, d_dzosum, d_alpha=None, stream=None):
    """cdfzonal_sum of a device-resident record, enqueued on `stream` (a torch stream or handle; None: the library's):
    d_zv (nk,ny,nx) f32, d_alpha (ny) f32 or None, into d_dzosum (nb,nk,ny) f64 -- torch CUDA tensors or device addresses."""
    p = _plans.get("zonal", {})
    _chk(load().cdfzonal_gpu_sum_device(_dev(d_zv, "d_zv", p.get("n3"), "float32"), _dev(d_alpha, "d_alpha", p.get("ny"), "float32"),
                                        _dev(d_dzosum, "d_dzosum", p.get("nout"), "float64"), C.c_void_p(stream_handle(stream))),
         "cdfzonal_gpu_sum_device")


def cdfzonal_mean_device(d_zv, d_dzomean, zspval=0.0, lmax=False, d_rzomax=None, d_rzomin=None, stream=None):
    """cdfzonal_mean of a device-resident record into d_dzomean (nb,nk,ny) f64 and, with lmax, d_rzomax / d_rzomin
    (nb,nk,ny) f32."""
    p = _plans.get("zonal", {})
    n = p.get("nout")
    _chk(load().cdfzonal_gpu_mean_device(_dev(d_zv, "d_zv", p.get("n3"), "float32"), float(zspval), int(bool(lmax)),
                                         _dev(d_dzomean, "d_dzomean", n, "float64"), _dev(d_rzomax, "d_rzomax", n, "float32"),
                                         _dev(d_rzomin, "d_rzomin", n, "float32"), C.c_void_p(stream_handle(stream))),
         "cdfzonal_gpu_mean_device")


# The record pipelines of the sibling tools (cdfzonal_gpu_submit_* / cdfmhst_gpu_submit* / cdftransig_gpu_submit): the library
# reads a submitted record's host arrays until the matching fetch (or cdftransig_gpu_wait) returns, so the arrays handed to
# the C call -- converted copies included -- are held here per slot until then (DESIGN.md section 0).
_held: dict = {}


def _drop(tool=None):
    """Setup, teardown and finalize wait for the records in flight and forget them: their arrays are released."""
    for k in [k for k in _held if tool is None or k[0] == tool]:
        del _held[k]


def cdfzonal_submit_sum(slot: int, zv, alpha=None):
    """cdfzonal_sum of one record on pipeline slot `slot` (0 .. nslots()-1); the result comes from cdfzonal_fetch."""
    zv = _rec(zv)
    al = _c32(alpha) if alpha is not None else None
    _chk(load().cdfzonal_gpu_submit_sum(int(slot), _ptr(zv), _ptr(al)), "cdfzonal_gpu_submit_sum")
    _held[("zonal", int(slot))] = (False, (zv, al))


def cdfzonal_submit_mean(slot: int, zv, zspval=0.0, lmax=False):
    zv = _rec(zv)
    _chk(load().cdfzonal_gpu_submit_mean(int(slot), _ptr(zv), float(zspval), int(bool(lmax))), "cdfzonal_gpu_submit_mean")
    _held[("zonal", int(slot))] = (True, bool(lmax), (zv,))


def cdfzonal_fetch(slot: int, shape):
    """-> what the synchronous call of the slot's submit returns: dzosum, or (dzomean, rzomax, rzomin)."""
    rec = _held.get(("zonal", int(slot)))
    mean, lmax = (rec[0], rec[1]) if rec is not None and rec[0] else (False, False)
    out = np.empty(shape, np.float64)
    zmax = np.empty(shape, np.float32) if lmax else None
    zmin = np.empty(shape, np.float32) if lmax else None
    _chk(load().cdfzonal_gpu_fetch(int(slot), _ptr(out), _ptr(zmax), _ptr(zmin)), "cdfzonal_gpu_fetch")
    _held.pop(("zonal", int(slot)), None)
    return (out, zmax, zmin) if mean else out


def cdfzonal_kernel_ms() -> float:
    ms = C.c_float()
    _chk(load().cdfzonal_gpu_kernel_ms(C.byref(ms)), "cdfzonal_gpu_kernel_ms")
    return ms.value


def cdfzonal_teardown():
    _chk(load().cdfzonal_gpu_teardown(), "cdfzonal_gpu_teardown")
    _drop("zonal")
    _plans.pop("zonal", None)


def cdfmhst_setup(e1v, e3v, vmask1, atl=None, pac=None, ind=None):
    e1v, e3v, vmask1 = _c32(e1v), _c32(e3v), _c32(vmask1)
    nz, ny, nx = e3v.shape
    a, p, i = (_c32(x) if x is not None else None for x in (atl, pac, ind))
    _chk(load().cdfmhst_gpu_setup(nx, ny, nz, _ptr(e1v), _ptr(e3v), _ptr(vmask1), _ptr(a), _ptr(p), _ptr(i)), "cdfmhst_gpu_setup")
    _drop("mhst")
    _plans["mhst"] = dict(n3=nz * ny * nx, nz=nz, ny=ny)
    return nz, ny


def cdfmhst_record(zvt, zvs, dims, zdim=False):
    """zvt, zvs (nz,ny,nx) f32 -> heat, salt (nlev,4,ny) f64 raw zonal sums (glo, atl, pac, ind)."""
    zvt, zvs = _rec(zvt), _rec(zvs)
    nz, ny = dims
    nlev = nz if zdim else 1
    heat, salt = np.empty((nlev, 4, ny), np.float64), np.empty((nlev, 4, ny), np.float64)
    _chk(load().cdfmhst_gpu_record(_ptr(zvt), _ptr(zvs), int(zdim), _ptr(heat), _ptr(salt)), "cdfmhst_gpu_record")
    return heat, salt


def cdfmhst_record_vts(zv, zt, zs, dims, zdim=False):
    """-v/-t[-s] mode: zv, zt, zs (nz,ny,nx) as read (f32, or int16 per set_sibling_input); the device forms the V-point
    products (cdfmhst.f90:313-323) and proceeds as cdfmhst_record."""
    zv, zt, zs = _rec(zv), _rec(zt), _rec(zs)
    nz, ny = dims
    nlev = nz if zdim else 1
    heat, salt = np.empty((nlev, 4, ny), np.float64), np.empty((nlev, 4, ny), np.float64)
    _chk(load().cdfmhst_gpu_record_vts(_ptr(zv), _ptr(zt), _ptr(zs), int(zdim), _ptr(heat), _ptr(salt)), "cdfmhst_gpu_record_vts")
    return heat, salt


def _mhst_device_args(records, d_heat, d_salt, zdim):
    p = _plans.get("mhst")
    nout = (p["nz"] if zdim else 1) * 4 * p["ny"] if p else None
    n3 = p["n3"] if p else None
    return ([_dev(a, name, n3, "float32") for name, a in records]
            + [_dev(d_heat, "d_heat", nout, "float64"), _dev(d_salt, "d_salt", nout, "float64")])


def cdfmhst_record_device(d_zvt, d_zvs, d_heat, d_salt, zdim=False, stream=None):
    """cdfmhst_record of device-resident records d_zvt, d_zvs (nz,ny,nx) f32 into d_heat, d_salt (nlev,4,ny) f64, enqueued
    on `stream` (torch CUDA tensors or device addresses)."""
    zvt, zvs, heat, salt = _mhst_device_args((("d_zvt", d_zvt), ("d_zvs", d_zvs)), d_heat, d_salt, zdim)
    _chk(load().cdfmhst_gpu_record_device(zvt, zvs, int(bool(zdim)), heat, salt, C.c_void_p(stream_handle(stream))),
         "cdfmhst_gpu_record_device")


def cdfmhst_record_vts_device(d_zv, d_zt, d_zs, d_heat, d_salt, zdim=False, stream=None):
    """cdfmhst_record_vts of device-resident records d_zv, d_zt, d_zs (nz,ny,nx) f32, enqueued on `stream`."""
    zv, zt, zs, heat, salt = _mhst_device_args((("d_zv", d_zv), ("d_zt", d_zt), ("d_zs", d_zs)), d_heat, d_salt, zdim)
    _chk(load().cdfmhst_gpu_record_vts_device(zv, zt, zs, int(bool(zdim)), heat, salt, C.c_void_p(stream_handle(stream))),
         "cdfmhst_gpu_record_vts_device")


def cdfmhst_submit(slot: int, zvt, zvs, zdim=False):
    zvt, zvs = _rec(zvt), _rec(zvs)
    _chk(load().cdfmhst_gpu_submit(int(slot), _ptr(zvt), _ptr(zvs), int(bool(zdim))), "cdfmhst_gpu_submit")
    _held[("mhst", int(slot))] = (bool(zdim), (zvt, zvs))


def cdfmhst_submit_vts(slot: int, zv, zt, zs, zdim=False):
    zv, zt, zs = _rec(zv), _rec(zt), _rec(zs)
    _chk(load().cdfmhst_gpu_submit_vts(int(slot), _ptr(zv), _ptr(zt), _ptr(zs), int(bool(zdim))), "cdfmhst_gpu_submit_vts")
    _held[("mhst", int(slot))] = (bool(zdim), (zv, zt, zs))


def cdfmhst_fetch(slot: int, dims):
    """-> heat, salt (nlev,4,ny) of the slot's record, as cdfmhst_record returns them."""
    rec = _held.get(("mhst", int(slot)))
    nz, ny = dims
    nlev = nz if rec is not None and rec[0] else 1
    heat, salt = np.empty((nlev, 4, ny), np.float64), np.empty((nlev, 4, ny), np.float64)
    _chk(load().cdfmhst_gpu_fetch(int(slot), _ptr(heat), _ptr(salt)), "cdfmhst_gpu_fetch")
    _held.pop(("mhst", int(slot)), None)
    return heat, salt


def cdfmhst_kernel_ms() -> float:
    ms = C.c_float()
    _chk(load().cdfmhst_gpu_kernel_ms(C.byref(ms)), "cdfmhst_gpu_kernel_ms")
    return ms.value


def cdfmhst_teardown():
    _chk(load().cdfmhst_gpu_teardown(), "cdfmhst_gpu_teardown")
    _drop("mhst")
    _plans.pop("mhst", None)


# ---- cdftransig_xy3d (src/cdftransig_xy3d.f90) -------------------------------------------------------------------
TRANSIG_CODES = {   # -code presets (cdftransig_xy3d.f90:188-197): pref, nbins, ds1min, ds1scal, ds1zoom, ds1scalmin
    "0": (0.0, 101, 23.0, 0.03, 999.0, 999.0), "1000": (1000.0, 93, 24.2, 0.10, 32.3, 0.05),
    "1000-acc": (1000.0, 88, 24.5, 0.10, 999.0, 999.0), "2000": (2000.0, 174, 29.0, 0.05, 999.0, 999.0),
}


def transig_bins(nbins, ds1min, ds1scal, ds1zoom=999.0, ds1scalmin=999.0):
    """Host side of cdftransig_xy3d.f90:213,229-262: bin centres dsigma(nbins), edges dsig_edge(nbins+1), the step -> bin
    table itab(nsigmax) (1-based bins, 0 = no bin) and the step MIN(ds1scalmin, ds1scal), all in REAL(8)."""
    ds1scalmin = min(float(ds1scalmin), float(ds1scal))
    dsigma = np.empty(nbins, np.float64)
    ijtrans = 0
    for ji in range(1, nbins + 1):
        test = ds1min + (ji - 0.5) * ds1scal
        if test > ds1zoom:
            if ijtrans == 0:
                ijtrans = ji
            dsigma[ji - 1] = ds1zoom + (ji - ijtrans + 0.5) * ds1scalmin
        else:
            dsigma[ji - 1] = test
    edge = np.empty(nbins + 1, np.float64)
    edge[0] = ds1min
    for ji in range(2, nbins + 1):
        edge[ji - 1] = 0.5 * (dsigma[ji - 1] + dsigma[ji - 2])
    edge[nbins] = edge[nbins - 1] + ds1scalmin
    x = (edge[nbins] - edge[0]) / ds1scalmin
    nsigmax = int(np.floor(abs(x) + 0.5)) * (1 if x >= 0 else -1)       # NINT
    itab = np.zeros(max(nsigmax, 0), np.int32)
    for ji in range(1, nsigmax + 1):
        test = ds1min + (ji - 0.5) * ds1scalmin
        for jj in range(1, nbins + 1):
            if edge[jj - 1] < test <= edge[jj]:
                itab[ji - 1] = jj
    return dsigma, edge, itab, ds1scalmin


def cdftransig_setup(e2u, e1v, e3u, e3v, nz, nbins, pref, ds1min, ds1scalmin, itab, lperio=False, teos10=False):
    """e2u, e1v (ny,nx); e3u, e3v (nz-1,ny,nx) or None (-vvl).  Zeroes the device accumulators."""
    e2u, e1v = _c32(e2u), _c32(e1v)
    ny, nx = e1v.shape
    e3u = _c32(e3u) if e3u is not None else None
    e3v = _c32(e3v) if e3v is not None else None
    assert e3u is None or (e3u.shape == (nz - 1, ny, nx) and e3v.shape == (nz - 1, ny, nx))
    it = np.ascontiguousarray(itab, np.int32)
    _chk(load().cdftransig_gpu_setup(nx, ny, nz, int(nbins), float(pref), int(teos10), float(ds1min), float(ds1scalmin),
                                     int(it.size), _ptr(it), _ptr(e2u), _ptr(e1v), _ptr(e3u), _ptr(e3v), int(lperio)),
         "cdftransig_gpu_setup")
    _drop("transig")
    _plans["transig"] = dict(n3=(nz - 1) * ny * nx, nacc=int(nbins) * ny * nx)
    return nbins, ny, nx


def cdftransig_record(zu, zv, zt, zs, set_masks, e3u_vvl=None, e3v_vvl=None):
    zu, zv, zt, zs = _rec(zu), _rec(zv), _rec(zt), _rec(zs)
    eu = _rec(e3u_vvl) if e3u_vvl is not None else None
    ev = _rec(e3v_vvl) if e3v_vvl is not None else None
    _chk(load().cdftransig_gpu_record(_ptr(zu), _ptr(zv), _ptr(zt), _ptr(zs), _ptr(eu), _ptr(ev), int(bool(set_masks))),
         "cdftransig_gpu_record")


def cdftransig_submit(slot: int, zu, zv, zt, zs, set_masks, e3u_vvl=None, e3v_vvl=None):
    """cdftransig_record as a pipeline on slot `slot` (0 .. nslots of init - 1, first device); the arrays are held until
    cdftransig_wait(slot) or cdftransig_fetch."""
    arrs = [_rec(zu), _rec(zv), _rec(zt), _rec(zs), _rec(e3u_vvl) if e3u_vvl is not None else None,
            _rec(e3v_vvl) if e3v_vvl is not None else None]
    _chk(load().cdftransig_gpu_submit(int(slot), *(_ptr(a) for a in arrs), int(bool(set_masks))), "cdftransig_gpu_submit")
    _held[("transig", int(slot))] = arrs


def cdftransig_wait(slot: int):
    _chk(load().cdftransig_gpu_wait(int(slot)), "cdftransig_gpu_wait")
    _held.pop(("transig", int(slot)), None)


def cdftransig_fetch(shape):
    du, dv = np.empty(shape, np.float64), np.empty(shape, np.float64)
    _chk(load().cdftransig_gpu_fetch(_ptr(du), _ptr(dv)), "cdftransig_gpu_fetch")
    _drop("transig")
    return du, dv


def cdftransig_record_device(d_zu, d_zv, d_zt, d_zs, set_masks, d_e3u_vvl=None, d_e3v_vvl=None, stream=None):
    """cdftransig_record of a device-resident frame (nz-1,ny,nx) f32, enqueued on `stream`; it accumulates in call order with
    the frames of cdftransig_record / cdftransig_submit."""
    n3 = _plans.get("transig", {}).get("n3")
    arrs = [_dev(a, name, n3, "float32") for name, a in (("d_zu", d_zu), ("d_zv", d_zv), ("d_zt", d_zt), ("d_zs", d_zs),
                                                        ("d_e3u_vvl", d_e3u_vvl), ("d_e3v_vvl", d_e3v_vvl))]
    _chk(load().cdftransig_gpu_record_device(*arrs, int(bool(set_masks)), C.c_void_p(stream_handle(stream))),
         "cdftransig_gpu_record_device")


def cdftransig_fetch_device(d_dusigsig, d_dvsigsig, stream=None):
    """The raw sums (nbins,ny,nx) f64 into device buffers, enqueued on `stream` after every frame so far."""
    n = _plans.get("transig", {}).get("nacc")
    _chk(load().cdftransig_gpu_fetch_device(_dev(d_dusigsig, "d_dusigsig", n, "float64"), _dev(d_dvsigsig, "d_dvsigsig", n, "float64"),
                                            C.c_void_p(stream_handle(stream))), "cdftransig_gpu_fetch_device")


def cdftransig_kernel_ms() -> float:
    ms = C.c_float()
    _chk(load().cdftransig_gpu_kernel_ms(C.byref(ms)), "cdftransig_gpu_kernel_ms")
    return ms.value


def cdftransig_teardown():
    _chk(load().cdftransig_gpu_teardown(), "cdftransig_gpu_teardown")
    _drop("transig")
    _plans.pop("transig", None)


def cdfsigtrp_section(eu, de3, ddepu, gdepw, zu, zt, zs, zmask, nk, dsigma_min, dsigma_max, nbins, mode=0, refdep=0.0,
                      teos10=False, ddepw_brk=None):
    """One cdfsigtrp section on the device (src/cdfsigtrp.f90:559-627) -> dict(dsigma_lev, dsig, dhiso, dwtrp, dwtrpbin,
    dtrpbin); arrays (npk, npts) C order = the reference's (npts,npk).  mode 0 sigmai(refdep), 1 neutral, 2 -temp."""
    eu, de3, zu, zt, zs, zmask = (_c32(x) for x in (eu, de3, zu, zt, zs, zmask))
    gdepw = _c32(gdepw) if gdepw is not None else None
    brk = _c32(ddepw_brk) if ddepw_brk is not None else None
    ddepu = np.ascontiguousarray(ddepu, np.float64)
    npk, npts = zu.shape
    assert ddepu.shape == (npk + 1, npts) and de3.shape == (npk, npts) and eu.shape == (npts,)
    out = dict(dsigma_lev=np.empty(nbins + 1, np.float64), dsig=np.empty((nk + 1, npts), np.float64),
               dhiso=np.empty((nbins + 1, npts), np.float64), dwtrp=np.empty((nbins + 1, npts), np.float64),
               dwtrpbin=np.empty((nbins, npts), np.float64), dtrpbin=np.empty(nbins, np.float64))
    _chk(load().cdfsigtrp_gpu_section(npts, npk, int(nk), _ptr(eu), _ptr(de3), _ptr(ddepu), _ptr(gdepw), _ptr(brk), _ptr(zu),
                                      _ptr(zt), _ptr(zs), _ptr(zmask), int(mode), float(refdep), int(teos10), float(dsigma_min),
                                      float(dsigma_max), int(nbins), _ptr(out["dsigma_lev"]), _ptr(out["dsig"]),
                                      _ptr(out["dhiso"]), _ptr(out["dwtrp"]), _ptr(out["dwtrpbin"]), _ptr(out["dtrpbin"])),
         "cdfsigtrp_gpu_section")
    return out


def cdfsigtrp_kernel_ms() -> float:
    ms = C.c_float()
    _chk(load().cdfsigtrp_gpu_kernel_ms(C.byref(ms)), "cdfsigtrp_gpu_kernel_ms")
    return ms.value


def cdfsigtrp_sections_setup(ijbox, gdept_1d, gdepw, dsigma_min, dsigma_max, nbins, e1v=None, e2u=None, e3u=None, e3v=None, e3w=None,
                             e3t_1d=None, e3w_1d=None, zspu=0.0, zspv=0.0, zsps=0.0, mode=0, refdep=0.0, teos10=False):
    """Plan of a section list for cdfsigtrp_sections_device: ijbox (nsec,4) imin imax jmin jmax (1-based F points, as in
    dens_section.dat); e1v, e2u (ny,nx) and e3u, e3v, e3w (npk,ny,nx) f32, or e3u = e3v = e3w = None with e3t_1d, e3w_1d
    (npk) for -full; gdept_1d, gdepw (npk).  mode 0 sigmai(refdep), 1 neutral, 2 -temp.  -> (dsigma_lev (nbins+1) f64,
    npts (nsec) int32, 0 for a skipped section)."""
    box = np.ascontiguousarray(ijbox, np.int32).reshape(-1, 4)
    nsec = box.shape[0]
    gdept_1d, gdepw = _c32(gdept_1d), _c32(gdepw)
    npk = gdepw.size
    e1v, e2u, e3u, e3v, e3w, e3t_1d, e3w_1d = (None if a is None else _c32(a) for a in (e1v, e2u, e3u, e3v, e3w, e3t_1d, e3w_1d))
    hz = next((a for a in (e1v, e2u) if a is not None), None)
    assert hz is not None and hz.ndim == 2, "e1v or e2u (ny,nx) is needed for the grid size"
    ny, nx = hz.shape
    assert all(a is None or a.shape == (ny, nx) for a in (e1v, e2u))
    assert all(a is None or a.shape == (npk, ny, nx) for a in (e3u, e3v, e3w))
    lev, npts = np.empty(int(nbins) + 1, np.float64), np.empty(nsec, np.int32)
    _chk(load().cdfsigtrp_gpu_sections_setup(nx, ny, npk, nsec, _ptr(box), _ptr(e1v), _ptr(e2u), _ptr(e3u), _ptr(e3v), _ptr(e3w),
                                             _ptr(e3t_1d), _ptr(e3w_1d), _ptr(gdept_1d), _ptr(gdepw), float(zspu), float(zspv),
                                             float(zsps), int(mode), float(refdep), int(teos10), float(dsigma_min), float(dsigma_max),
                                             int(nbins), _ptr(lev), _ptr(npts)), "cdfsigtrp_gpu_sections_setup")
    _plans["sigtrp"] = dict(n3=npk * ny * nx, nout=nsec * int(nbins), nsec=nsec)
    return lev, npts


def cdfsigtrp_sections_device(d_u, d_v, d_t, d_s, d_dtrpbin, d_nk=None, stream=None):
    """Every section of the plan on one device-resident record, enqueued on `stream` (a torch stream or handle; None: the
    library's): d_u, d_v, d_t, d_s (npk,ny,nx) f32 (d_u / d_v may be None when no section is meridional / zonal) ->
    d_dtrpbin (nsec,nbins) f64 in m3/s, d_nk (nsec) int32 or None -- torch CUDA tensors or device addresses."""
    p = _plans.get("sigtrp", {})
    n3 = p.get("n3")
    fields = [_dev(a, name, n3, "float32") for name, a in (("d_u", d_u), ("d_v", d_v), ("d_t", d_t), ("d_s", d_s))]
    _chk(load().cdfsigtrp_gpu_sections_device(*fields, _dev(d_dtrpbin, "d_dtrpbin", p.get("nout"), "float64"),
                                              _dev(d_nk, "d_nk", p.get("nsec"), "int32"), C.c_void_p(stream_handle(stream))),
         "cdfsigtrp_gpu_sections_device")


def cdfsigtrp_teardown():
    """Frees the single-section scratch and the sections plan, after the device calls that read it."""
    _chk(load().cdfsigtrp_gpu_teardown(), "cdfsigtrp_gpu_teardown")
    _plans.pop("sigtrp", None)
