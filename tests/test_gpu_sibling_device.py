"""cdfzonal, cdfmhst and cdftransig on device-resident fields (the *_device entry points of include/cdfgpu.h): the same
kernels on the caller's device pointers and stream.  Every result must equal the host-array call bit for bit, on the
library's stream and on a torch stream; cdftransig frames of every entry point accumulate in call order; the calls only
enqueue work and copy nothing between host and device."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from cdftools_b200 import lib, synth
from test_gpu_sibling_edges import K6_CFGS, exact_field, mhst_exact, transig_frames, zonal_exact

ROOT = Path(__file__).resolve().parent.parent
ERR_ARG, ERR_STATE, ERR_NODEVICE = 2, 3, 5
ZSP = -99999.0
FILL = -7.77e33   # what an output element holds when the call never wrote it
gpu = pytest.mark.gpu


def same(a, b):
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def out(shape, dtype):
    import torch
    return torch.full(shape, FILL, dtype=dtype, device="cuda")


@pytest.fixture(params=["library", "torch"])
def stream(request, gpu_lib):
    """None (the library's compute stream) or a torch stream; inputs made on torch's default stream are complete first."""
    import torch
    torch.cuda.synchronize()
    yield None if request.param == "library" else torch.cuda.Stream()
    torch.cuda.synchronize()


def on(st, fn):
    """Run fn on stream st (None: enqueued on the library's stream) and wait for the device."""
    import torch
    if st is None:
        fn(None)
    else:
        with torch.cuda.stream(st):
            fn(st)
    torch.cuda.synchronize()


# ---- 1. device == host, bit for bit -------------------------------------------------------------------------------------------
def check_zonal(case, st, nonfinite=False):
    import torch
    e1, e2, zm, mv, zv, alpha = case
    if nonfinite:   # in a row with mixed basin masks, and in rows of their own
        zv = zv.copy()
        zv.flat[[0, zv.size // 2, zv.size - 1]] = [np.inf, np.nan, -np.inf]
    shape = lib.cdfzonal_setup(e1, e2, zm, mv)
    try:
        d_zv, d_al = dev(zv), dev(alpha)
        for al, d_a in ((alpha, d_al), (None, None)):
            d_o = out(shape, torch.float64)
            on(st, lambda s: lib.cdfzonal_sum_device(d_zv, d_o, d_a, stream=s))
            assert same(d_o.cpu().numpy(), lib.cdfzonal_sum(zv, shape, al)), f"sum, alpha {al is not None}"
        for lmax in (False, True):
            d_o, d_mx, d_mn = out(shape, torch.float64), out(shape, torch.float32), out(shape, torch.float32)
            on(st, lambda s: lib.cdfzonal_mean_device(d_zv, d_o, ZSP, lmax, d_mx if lmax else None, d_mn if lmax else None,
                                                      stream=s))
            ref = lib.cdfzonal_mean(zv, shape, ZSP, lmax)
            assert same(d_o.cpu().numpy(), ref[0]), f"mean, lmax {lmax}"
            if lmax:
                assert same(d_mx.cpu().numpy(), ref[1]) and same(d_mn.cpu().numpy(), ref[2]), "max / min"
    finally:
        lib.cdfzonal_teardown()


ZONAL_NX = [1, 2, 3, 4, 5, 6, 7, 33, 1442, 4322]


@gpu
@pytest.mark.parametrize("nx", ZONAL_NX)
def test_zonal_widths(stream, nx):
    check_zonal(zonal_exact(nx, 3, 2, 3, nx), stream)


@gpu
@pytest.mark.parametrize("general", [None, 0.5], ids=["bits", "half"])
@pytest.mark.parametrize("nb", range(1, 9))
def test_zonal_basin_counts(stream, nb, general):
    check_zonal(zonal_exact(37, 5, 3, nb, 100 + nb, general), stream)


@gpu
@pytest.mark.parametrize("shape", [(33, 1, 4), (33, 4, 1), (1, 1, 1)], ids=["ny1", "nk1", "one-cell"])
def test_zonal_edge_shapes(stream, shape):
    nx, ny, nk = shape
    check_zonal(zonal_exact(nx, ny, nk, 5, nx * ny + nk), stream)


@gpu
@pytest.mark.parametrize("general", [None, 0.5], ids=["bits", "half"])
def test_zonal_nonfinite_cells(stream, general):
    check_zonal(zonal_exact(37, 6, 2, 3, 11, general), stream, nonfinite=True)


def check_mhst(nx, ny, nz, seed, st, basins=True, nonfinite=False):
    import torch
    e1v, e3v, v1, b3, zvt, zvs = mhst_exact(nx, ny, nz, seed)
    zv = exact_field((nz, ny, nx), nbits=5)
    zt = (exact_field((nz, ny, nx), nbits=6, offset=7) + np.float32(10.0)).astype(np.float32)
    zs = (exact_field((nz, ny, nx), nbits=6, offset=3) + np.float32(35.0)).astype(np.float32)
    if nonfinite:
        zvt.flat[[1, zvt.size // 3]] = [np.nan, np.inf]
        zt.flat[zt.size // 2] = -np.inf
        zs.flat[zs.size - 2] = np.nan
    kw = dict(zip(("atl", "pac", "ind"), b3)) if basins else {}
    dims = lib.cdfmhst_setup(e1v, e3v, v1, **kw)
    try:
        d = [dev(a) for a in (zvt, zvs, zv, zt, zs)]
        for zdim in (False, True):
            nlev = nz if zdim else 1
            for vts in (False, True):
                h, s_ = out((nlev, 4, ny), torch.float64), out((nlev, 4, ny), torch.float64)
                if vts:
                    on(st, lambda s: lib.cdfmhst_record_vts_device(d[2], d[3], d[4], h, s_, zdim, stream=s))
                    ref = lib.cdfmhst_record_vts(zv, zt, zs, dims, zdim)
                else:
                    on(st, lambda s: lib.cdfmhst_record_device(d[0], d[1], h, s_, zdim, stream=s))
                    ref = lib.cdfmhst_record(zvt, zvs, dims, zdim)
                assert same(h.cpu().numpy(), ref[0]) and same(s_.cpu().numpy(), ref[1]), f"zdim {zdim}, vts {vts}"
    finally:
        lib.cdfmhst_teardown()


@gpu
@pytest.mark.parametrize("nx", [1, 2, 3, 5, 7, 33, 257, 1442, 2049, 4097, 4322, 8192])
def test_mhst_widths(stream, nx):
    check_mhst(nx, 3, 4, nx, stream)


@gpu
@pytest.mark.parametrize("shape", [(5, 1, 3), (33, 4, 1), (1, 1, 2)], ids=["ny1", "one-level", "one-column"])
def test_mhst_edge_shapes(stream, shape):
    nx, ny, nz = shape
    check_mhst(nx, ny, nz, nx * ny * nz, stream, basins=False)


@gpu
def test_mhst_nonfinite_cells(stream):
    check_mhst(37, 5, 4, 3, stream, nonfinite=True)


TRANSIG_SHAPES = [synth.GRIDS["TINY"], synth.GRIDS["ODD"], (1, 4, 3), (3, 4, 3), (9, 1, 3), (11, 5, 2), (1442, 6, 12)]
TRANSIG_IDS = ["TINY", "ODD", "nx1", "nx3", "ny1", "nz2", "orca025-band"]


def transig_case(shape, cfg, vvl, nframes=3):
    pref, code, lperio, teos10 = cfg
    nx, ny, nz = shape
    e2u, e1v, e3u, e3v, frames = transig_frames(nx, ny, nz, nframes, nx * 7 + ny + nz)
    if vvl:   # every frame brings its own e3
        rng = np.random.default_rng(nx + ny)
        frames = [f + tuple((e * (1 + 0.1 * rng.random(e.shape))).astype(np.float32) for e in (e3u, e3v)) for f in frames]
    _, _, itab, scm = lib.transig_bins(*code)
    setup = (e2u, e1v, None if vvl else e3u, None if vvl else e3v, nz, code[0], pref, code[1], scm, itab, lperio, teos10)
    return setup, frames


def transig_host(setup, frames, nmask=2):
    shp = lib.cdftransig_setup(*setup)
    try:
        for n, f in enumerate(frames):
            lib.cdftransig_record(*f[:4], set_masks=n < nmask, e3u_vvl=f[4] if len(f) > 4 else None,
                                  e3v_vvl=f[5] if len(f) > 5 else None)
        return lib.cdftransig_fetch(shp)
    finally:
        lib.cdftransig_teardown()


@gpu
@pytest.mark.parametrize("vvl", [False, True], ids=["e3", "vvl"])
@pytest.mark.parametrize("cfg", K6_CFGS[:2], ids=["sigma0", "sigma1-perio"])
@pytest.mark.parametrize("shape", TRANSIG_SHAPES, ids=TRANSIG_IDS)
def test_transig_frames(stream, shape, cfg, vvl):
    """Three frames, masks set by the first two (two tags); -vvl frames with device e3.  fetch_device and fetch agree."""
    import torch
    setup, frames = transig_case(shape, cfg, vvl)
    ref = transig_host(setup, frames)
    shp = lib.cdftransig_setup(*setup)
    try:
        d_frames = [[dev(a) for a in f] for f in frames]
        du, dv = out(shp, torch.float64), out(shp, torch.float64)

        def run(s):
            for n, f in enumerate(d_frames):
                lib.cdftransig_record_device(*f[:4], n < 2, *f[4:], stream=s)
            lib.cdftransig_fetch_device(du, dv, stream=s)

        on(stream, run)
        host = lib.cdftransig_fetch(shp)
    finally:
        lib.cdftransig_teardown()
    for got in ((du.cpu().numpy(), dv.cpu().numpy()), host):
        assert same(got[0], ref[0]) and same(got[1], ref[1])
    assert np.isnan(ref[0]).any() and np.count_nonzero(ref[0]) > 0


# ---- 2. cdftransig: frames of every entry point in call order ----------------------------------------------------------------
@gpu
@pytest.mark.parametrize("vvl", [False, True], ids=["e3", "vvl"])
def test_transig_interleaved_entry_points(gpu_lib, vvl):
    """submit, record_device, submit, record, record_device, fetch_device, submit, fetch, fetch_device (library stream):
    every fetch equals the all-host frame loop over the frames before it, bit for bit."""
    import torch
    setup, frames = transig_case(synth.GRIDS["ODD"], K6_CFGS[1], vvl, nframes=6)
    refs = {n: transig_host(setup, frames[:n]) for n in (5, 6)}
    shp = lib.cdftransig_setup(*setup)
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    try:
        d = [[dev(a) for a in f] for f in frames]
        e3 = lambda n: dict(e3u_vvl=frames[n][4], e3v_vvl=frames[n][5]) if vvl else {}
        mid = (out(shp, torch.float64), out(shp, torch.float64))
        end = (out(shp, torch.float64), out(shp, torch.float64))
        with torch.cuda.stream(st):
            lib.cdftransig_submit(0, *frames[0][:4], set_masks=True, **e3(0))
            lib.cdftransig_record_device(*d[1][:4], True, *d[1][4:], stream=st)
            lib.cdftransig_submit(1, *frames[2][:4], set_masks=False, **e3(2))
            lib.cdftransig_wait(0)
            lib.cdftransig_wait(1)
            lib.cdftransig_record(*frames[3][:4], set_masks=False, **e3(3))
            lib.cdftransig_record_device(*d[4][:4], False, *d[4][4:], stream=st)
            torch.cuda._sleep(20_000_000)   # the copy is still queued when the next frame is submitted
            lib.cdftransig_fetch_device(*mid, stream=st)
            lib.cdftransig_submit(2, *frames[5][:4], set_masks=False, **e3(5))
        host = lib.cdftransig_fetch(shp)
        lib.cdftransig_fetch_device(*end)
        torch.cuda.synchronize()
    finally:
        lib.cdftransig_teardown()
    for got, ref in ((tuple(t.cpu().numpy() for t in mid), refs[5]), (host, refs[6]), (tuple(t.cpu().numpy() for t in end), refs[6])):
        assert same(got[0], ref[0]) and same(got[1], ref[1])
    assert not same(refs[5][0], refs[6][0])


# ---- 3. stream semantics, 4. no copies -----------------------------------------------------------------------------------
class Tools:
    """Plans of the three tools, two records of each on the device, one set of device outputs, the host results.
    enqueue(ins, s): every *_device call once on stream s -- zonal sum and mean -max, mhst and mhst _vts, one transig frame
    and fetch_device -- reading the records in `ins` (names of src[r]); KERNELS is how many kernels that launches."""
    KERNELS = 1 + 1 + 1 + 2 + 2

    def __init__(self):
        import torch
        e1, e2, zm, mv, zv, alpha = zonal_exact(1442, 6, 3, 3, 5)
        zrec = [zv, (np.float32(-2.0) * zv + np.float32(1.0)).astype(np.float32)]
        e1v, e3v, v1, b3, zvt, zvs = mhst_exact(1442, 5, 4, 9)
        mrec = [(zvt, zvs, zvs), (zvs, zvt, zvt)]   # (zvt, zvs) of K5, and (zv, zt, zs) of K5v from the same fields
        self.tsetup, frames = transig_case(synth.GRIDS["ODD"], K6_CFGS[1], False, nframes=2)
        tref = [transig_host(self.tsetup, frames[:n + 1], nmask=1) for n in range(2)]
        self.zshape = lib.cdfzonal_setup(e1, e2, zm, mv)
        mdims = lib.cdfmhst_setup(e1v, e3v, v1, *b3)
        self.tshape = lib.cdftransig_setup(*self.tsetup)
        self.alpha = dev(alpha)
        self.src = [dict(zv=dev(zrec[r]), vt=dev(mrec[r][0]), vs=dev(mrec[r][1]), vv=dev(mrec[r][2]),
                         **{k: dev(a) for k, a in zip(("tu", "tv", "tt", "ts"), frames[r])}) for r in range(2)]
        self.host = [dict(sum=(lib.cdfzonal_sum(zrec[r], self.zshape, alpha),), mean=lib.cdfzonal_mean(zrec[r], self.zshape, ZSP, True),
                          mhst=lib.cdfmhst_record(mrec[r][0], mrec[r][1], mdims),
                          vts=lib.cdfmhst_record_vts(mrec[r][2], mrec[r][0], mrec[r][1], mdims), transig=tref[r]) for r in range(2)]
        z, h = self.zshape, (1, 4, mdims[1])
        f8, f4 = torch.float64, torch.float32
        self.o = dict(sum=(out(z, f8),), mean=(out(z, f8), out(z, f4), out(z, f4)), mhst=(out(h, f8), out(h, f8)),
                      vts=(out(h, f8), out(h, f8)), transig=(out(self.tshape, f8), out(self.tshape, f8)))
        self.frames = 0

    def enqueue(self, ins, s):
        o = self.o
        lib.cdfzonal_sum_device(ins["zv"], o["sum"][0], self.alpha, stream=s)
        lib.cdfzonal_mean_device(ins["zv"], o["mean"][0], ZSP, True, o["mean"][1], o["mean"][2], stream=s)
        lib.cdfmhst_record_device(ins["vt"], ins["vs"], *o["mhst"], stream=s)
        lib.cdfmhst_record_vts_device(ins["vv"], ins["vt"], ins["vs"], *o["vts"], stream=s)
        lib.cdftransig_record_device(ins["tu"], ins["tv"], ins["tt"], ins["ts"], self.frames == 0, stream=s)
        lib.cdftransig_fetch_device(*o["transig"], stream=s)
        self.frames += 1

    def check(self, r):
        """The outputs hold the results of record r (and the transig sums of frames 0..r)."""
        for k, ref in self.host[r].items():
            for got, want in zip(self.o[k], ref):
                assert same(got.cpu().numpy(), want), (k, r)

    def close(self):
        import torch
        torch.cuda.synchronize()
        lib.cdfzonal_teardown()
        lib.cdfmhst_teardown()
        lib.cdftransig_teardown()


@pytest.fixture
def tools(gpu_lib):
    import torch
    t = Tools()
    torch.cuda.synchronize()
    yield t
    t.close()


@gpu
def test_inputs_from_the_kernel_just_before(tools):
    """Each record is written by a torch kernel on the same stream right before the call, behind a ~10 ms sleep, with no
    synchronisation in between: the calls read what that kernel wrote."""
    import torch
    bufs = {k: torch.zeros_like(v) for k, v in tools.src[0].items()}
    torch.cuda.synchronize()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        torch.cuda._sleep(20_000_000)
        for k, b in bufs.items():
            b.copy_(tools.src[0][k])
        tools.enqueue(bufs, st)
    torch.cuda.synchronize()
    tools.check(0)


@gpu
def test_calls_only_enqueue(tools):
    """With the stream held by a sleep the calls return at once: the stream is still busy afterwards."""
    import torch
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        tools.enqueue(tools.src[0], st)   # first calls: the _vts scratch and the EOS table are in place afterwards
    torch.cuda.synchronize()
    with torch.cuda.stream(st):
        torch.cuda._sleep(400_000_000)   # ~0.2 s
        tools.enqueue(tools.src[1], st)
        busy = not st.query()
    torch.cuda.synchronize()
    assert busy
    tools.check(1)


@gpu
@pytest.mark.parametrize("library_stream", [False, True], ids=["torch", "library"])
def test_back_to_back_calls_leave_the_second_result(tools, library_stream):
    import torch
    st = None if library_stream else torch.cuda.Stream()
    on(st, lambda s: (tools.enqueue(tools.src[0], s), tools.enqueue(tools.src[1], s)))
    tools.check(1)


@gpu
def test_no_host_device_copies(tools):
    """A trace over device calls only: kernels, no HtoD / DtoH memcpy; cdfgpu_launch_count counts every kernel."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    st = torch.cuda.Stream()
    n0 = lib.launch_count()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        on(st, lambda s: (tools.enqueue(tools.src[0], s), tools.enqueue(tools.src[1], s)))
    assert lib.launch_count() - n0 == 2 * Tools.KERNELS
    names = [e.name for e in prof.events()]
    for k in ("zonal_rows_kernel", "mhst_rows_kernel", "mhst_vpoint_kernel", "transig_dens_kernel", "transig_scatter_kernel"):
        assert any(k in n for n in names), f"{k} not in the trace"
    copies = [n for n in names if "HtoD" in n or "DtoH" in n]
    assert not copies, copies
    tools.check(1)
    with profile(activities=[ProfilerActivity.CUDA]) as control:   # what a copy looks like in such a trace
        torch.ones(4).cuda()
        torch.cuda.synchronize()
    assert any("HtoD" in e.name for e in control.events())


# ---- 5. errors -------------------------------------------------------------------------------------------------------------
USES = {"zonal_sum": ("zv", "al", "zo"), "zonal_mean": ("zv", "zo", "mx", "mn"), "mhst": ("vt", "vs", "h", "s"),
        "mhst_vts": ("vv", "vt", "vs", "h", "s"), "transig": ("tu", "tv", "tt", "ts"), "transig_fetch": ("du", "dv")}
USES_ALL = sorted({k for v in USES.values() for k in v})


def each_call(t, a=None):
    """Every *_device entry point once, on tensors or addresses from t (name -> array): a dict name -> thunk."""
    a = a or {}
    g = lambda k: a.get(k, t[k])
    return {
        "zonal_sum": lambda: lib.cdfzonal_sum_device(g("zv"), g("zo"), g("al")),
        "zonal_mean": lambda: lib.cdfzonal_mean_device(g("zv"), g("zo"), ZSP, True, g("mx"), g("mn")),
        "mhst": lambda: lib.cdfmhst_record_device(g("vt"), g("vs"), g("h"), g("s")),
        "mhst_vts": lambda: lib.cdfmhst_record_vts_device(g("vv"), g("vt"), g("vs"), g("h"), g("s")),
        "transig": lambda: lib.cdftransig_record_device(g("tu"), g("tv"), g("tt"), g("ts"), True),
        "transig_fetch": lambda: lib.cdftransig_fetch_device(g("du"), g("dv")),
    }


def arrays(tools):
    s, o = tools.src[0], tools.o
    return dict(zv=s["zv"], al=tools.alpha, zo=o["mean"][0], mx=o["mean"][1], mn=o["mean"][2], vt=s["vt"], vs=s["vs"], vv=s["vv"],
                h=o["mhst"][0], s=o["mhst"][1], tu=s["tu"], tv=s["tv"], tt=s["tt"], ts=s["ts"], du=o["transig"][0], dv=o["transig"][1])


def code_of(thunk):
    with pytest.raises(lib.CdfGpuError) as ei:
        thunk()
    return ei.value.code


@gpu
def test_errors(tools):
    import torch
    t = arrays(tools)
    # a view 4 bytes into a larger allocation: right size, dtype and device, not 16-byte aligned
    off = {k: torch.empty(v.numel() + 1, dtype=v.dtype, device="cuda")[1:].view(v.shape) for k, v in t.items()}
    for name in USES:
        for k in USES[name]:
            assert code_of(each_call(t, {k: off[k]})[name]) == ERR_ARG, (name, k, lib.load().cdfgpu_last_error())
    # null required pointers, straight through the C ABI
    L, p = lib.load(), lambda k: t[k].data_ptr()
    assert L.cdfzonal_gpu_sum_device(None, p("al"), p("zo"), None) == ERR_ARG
    assert L.cdfzonal_gpu_mean_device(p("zv"), ZSP, 1, p("zo"), None, p("mn"), None) == ERR_ARG
    assert L.cdfmhst_gpu_record_device(p("vt"), None, 0, p("h"), p("s"), None) == ERR_ARG
    assert L.cdfmhst_gpu_record_vts_device(p("vv"), p("vt"), p("vs"), 0, p("h"), None, None) == ERR_ARG
    assert L.cdftransig_gpu_record_device(p("tu"), p("tv"), None, p("ts"), None, None, 1, None) == ERR_ARG
    assert L.cdftransig_gpu_fetch_device(p("du"), None, None) == ERR_ARG
    # the wrappers check tensors before the C call
    bad = {"zv": t["zv"].double(), "zo": t["zo"][:-1], "vt": t["vt"].cpu(), "h": t["h"].float(), "tu": t["tu"][..., :-1],
           "du": t["du"].transpose(1, 2), "al": t["al"][:-1], "mx": t["mx"].double()}
    for name in USES:
        for k, v in bad.items():
            if k in USES[name]:
                with pytest.raises(ValueError):
                    each_call(t, {k: v})[name]()
    with pytest.raises(ValueError):
        lib.cdfzonal_sum_device(t["zv"].cpu().numpy(), t["zo"])
    tools.close()   # before setup (the fixture's teardown of the empty plans is harmless)
    for name, call in each_call(t).items():
        assert code_of(call) == ERR_STATE, name


@gpu
def test_two_devices_refuse(gpu_lib):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    t = {k: 256 for k in USES_ALL}
    lib.finalize()
    try:
        lib.init_multi(2, "time", 3)
        for name, call in each_call(t).items():
            assert code_of(call) == ERR_STATE, name
            assert "one device" in lib.load().cdfgpu_last_error().decode()
    finally:
        lib.finalize()
        lib.init(0, 3)


# ---- 6. no device ------------------------------------------------------------------------------------------------------------
_NO_DEVICE = """
import sys
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, sys.argv[2])
from cdftools_b200 import lib
from test_gpu_sibling_device import USES_ALL, each_call
for name, call in each_call({k: 256 for k in USES_ALL}).items():
    try:
        call()
        sys.exit(name + " succeeded without a device")
    except lib.CdfGpuError as e:
        assert e.code == 5, (name, e.code)   # CDFGPU_ERR_NODEVICE
"""


def test_device_entry_points_without_a_device():
    """In a process that sees no device every *_device entry point fails with CDFGPU_ERR_NODEVICE (no CPU fallback)."""
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE, str(ROOT), str(ROOT / "tests")], capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stdout + r.stderr


