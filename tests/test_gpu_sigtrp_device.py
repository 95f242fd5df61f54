"""cdfsigtrp on device-resident fields (cdfsigtrp_gpu_sections_setup / _device): a list of dens_section.dat boxes cut from
whole U, V, T, S records and prepared on the device, every section in one batch of launches.  Each section's row must equal
the oracle fed with the slices tests/util.py cuts and oracle.sigtrp_prepare prepares, the host ABI call on those slices and
the command-line twin, bit for bit; nk must equal the oracle's.  The calls only enqueue work and copy nothing between host
and device."""
import os
import re
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
from scipy.io import netcdf_file

from cdftools_b200 import lib, ncfiles, synth
from test_sigtrp import SETTINGS
from util import sigtrp_expected

ROOT = Path(__file__).resolve().parent.parent
ERR_ARG, ERR_STATE, ERR_NODEVICE = 2, 3, 5
FILL = -7.77e33
gpu = pytest.mark.gpu
f32 = np.float32

# boxes whose fields the tests overwrite: every level all land (nk = 1), every level with ocean (nk = npk)
ALL_LAND, NO_LAND = (20, 24, 2, 2), (30, 30, 4, 7)


def section_list(nx, ny):
    return [(2, nx - 3, ny // 2, ny // 2),   # zonal
            (nx // 3, nx // 3, 1, ny - 2),   # meridional
            (3, 10, 2, 5),                   # oblique: skipped
            (5, 5, 4, 4),                    # no column: skipped
            (7, 8, 3, 3),                    # one column
            (1, nx, ny - 1, ny - 1),         # zonal on the last valid row, up to the last column
            (nx - 1, nx - 1, 0, ny),         # meridional on the last valid column, every row
            ALL_LAND, NO_LAND,
            (10, 10, 6, 2)]                  # jmax < jmin: skipped


def npts_of(sec):
    imin, imax, jmin, jmax = sec
    n = jmax - jmin if imin == imax else imax - imin if jmin == jmax else 0
    return max(n, 0)


def fields(m, spval=0.0, boxes=True):
    """U, V, T, S (npk,ny,nx) f32 as the gridU / gridV / gridT writers make their first record; land holds spval."""
    u = (synth.make_v_record(m, 500) * m.umask).astype(f32)
    if spval:
        u = np.where(m.umask.astype(bool), u, f32(spval)).astype(f32)
    v = synth.make_v_record(m, 0, spval=spval or None)
    t, s = synth.make_ts_record(m, 0, spval=spval or None)
    t, s = t.copy(), s.copy()
    if boxes:
        s[:, 1:3, 20:24] = spval        # ALL_LAND: rows 2-3, columns 21-24 (1-based)
        s[:, 4:7, 29:31] = f32(34.5)    # NO_LAND: rows 5-7, columns 30-31
        t[:, 4:7, 29:31] = f32(4.0)
    return u, v, t, s


def mesh_arrays(m, full=False):
    e3w_1d, e3w = ncfiles.e3w_fields(m)
    kw = dict(e1v=m.e1v, e2u=(m.e1u * f32(0.9)).astype(f32), gdept_1d=m.gdept_1d, gdepw=m.gdepw_1d)
    if full:
        kw.update(e3t_1d=m.e3t_1d, e3w_1d=e3w_1d)
    else:
        kw.update(e3u=(m.e3v_0 * f32(1.01)).astype(f32), e3v=m.e3v_0, e3w=e3w)
    return kw


def cut(m, u, v, t, s, sec, full):
    """The section's slices as util.sigtrp_expected cuts them; -full: e3t_1d / e3w_1d columns (cdfsigtrp_main.cpp -full)."""
    imin, imax, jmin, jmax = sec
    e3w_1d, e3w = ncfiles.e3w_fields(m)
    if imin == imax:
        rows, i0 = slice(jmin, jmax), imin - 1
        c = lambda a, i: np.ascontiguousarray(a[:, rows, i])
        eu, de3 = (m.e1u * f32(0.9)).astype(f32)[rows, i0].copy(), c((m.e3v_0 * f32(1.01)).astype(f32), i0)
        raw = dict(e3w_a=c(e3w, i0), e3w_b=c(e3w, i0 + 1), zu=c(u, i0), zs_a=c(s, i0), zs_b=c(s, i0 + 1), zt_a=c(t, i0), zt_b=c(t, i0 + 1))
    else:
        cols, j0 = slice(imin, imax), jmin - 1
        c = lambda a, j: np.ascontiguousarray(a[:, j, cols])
        eu, de3 = m.e1v[j0, imin - 1:imax - 1].copy(), c(m.e3v_0, j0)
        raw = dict(e3w_a=c(e3w, j0), e3w_b=c(e3w, j0 + 1), zu=c(v, j0), zs_a=c(s, j0), zs_b=c(s, j0 + 1), zt_a=c(t, j0), zt_b=c(t, j0 + 1))
    if full:
        npts = eu.size
        rep = lambda a: np.repeat(a.astype(f32)[:, None], npts, axis=1)
        de3, raw["e3w_a"], raw["e3w_b"] = rep(m.e3t_1d), rep(e3w_1d), rep(e3w_1d)
    return eu, de3, raw, imin == imax


def references(oracle_mod, m, flds, sec, setting, spval, full):
    """(oracle (p, o), host ABI dtrpbin) for one section."""
    mode, refdep, teos10, smin, smax, nbins = setting
    kw = dict(mode=mode, refdep=refdep, teos10=teos10)
    eu, de3, raw, merid = cut(m, *flds, sec, full)
    p = oracle_mod.sigtrp_prepare(m.gdept_1d[0], raw["e3w_a"], raw["e3w_b"], raw["zu"], spval, raw["zs_a"], raw["zs_b"], spval,
                                  raw["zt_a"], raw["zt_b"], merid=merid)
    args = (eu, de3, p["ddepu"], m.gdepw_1d.astype(f32), p["zu"], p["zt"], p["zs"], p["zmask"], p["nk"], smin, smax, nbins)
    if full:
        ref = (p, oracle_mod.sigtrp_section(*args, **kw))
    else:
        ref = sigtrp_expected(oracle_mod, m, *flds, sec, smin, smax, nbins, spval=spval, **kw)
        assert ref[0]["nk"] == p["nk"]
    host = lib.cdfsigtrp_section(*args, **kw)["dtrpbin"]
    return ref, host


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run_device(flds, nsec, nbins, stream=None):
    """One sections_device call on device copies of flds -> (dtrpbin (nsec,nbins), nk (nsec)) on the host."""
    import torch
    d = [dev(a) for a in flds]
    out = torch.full((nsec, nbins), FILL, dtype=torch.float64, device="cuda")
    nk = torch.full((nsec,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    lib.cdfsigtrp_sections_device(*d, out, nk, stream=stream)
    torch.cuda.synchronize()
    return out.cpu().numpy(), nk.cpu().numpy()


def setup(m, secs, setting, spval=0.0, full=False):
    mode, refdep, teos10, smin, smax, nbins = setting
    return lib.cdfsigtrp_sections_setup(np.array(secs), dsigma_min=smin, dsigma_max=smax, nbins=nbins, zspu=spval, zspv=spval,
                                        zsps=spval, mode=mode, refdep=refdep, teos10=teos10, **mesh_arrays(m, full))


def check(oracle_mod, m, flds, secs, setting, spval=0.0, full=False, nk_cases=True):
    nbins = setting[5]
    lev, npts = setup(m, secs, setting, spval, full)
    assert list(npts) == [npts_of(s) for s in secs]
    got, nk = run_device(flds, len(secs), nbins)
    for r, sec in enumerate(secs):
        if npts[r] == 0:
            assert np.all(got[r] == 0.0) and nk[r] == 0, sec
            continue
        (p, o), host = references(oracle_mod, m, flds, sec, setting, spval, full)
        assert np.array_equal(lev, o["dsigma_lev"])
        assert np.array_equal(got[r], o["dtrpbin"], equal_nan=True), (sec, np.nanmax(np.abs(got[r] - o["dtrpbin"])))
        assert np.array_equal(got[r], host, equal_nan=True), sec
        assert nk[r] == p["nk"], (sec, nk[r], p["nk"])
        if nk_cases and sec == ALL_LAND:
            assert p["nk"] == 1
        if nk_cases and sec == NO_LAND:
            assert p["nk"] == m.nz and not p["found"]
    return got


@pytest.fixture
def sigtrp(gpu_lib):
    import torch
    torch.cuda.synchronize()
    yield lib
    lib.cdfsigtrp_teardown()


# ---- 1, 2. every section against the oracle and the host ABI call ---------------------------------------------------------
@gpu
@pytest.mark.parametrize("full", [False, True], ids=["e3", "full"])
@pytest.mark.parametrize("setting", SETTINGS, ids=["sigma0", "sigma2000", "neutral", "temp", "teos10"])
@pytest.mark.parametrize("grid", ["SMALL", "ODD"])
def test_sections_match_oracle_and_host_call(sigtrp, oracle_mod, grid, setting, full):
    if full and setting is not SETTINGS[0] and setting is not SETTINGS[3]:
        pytest.skip("-full: sigma0 and -temp cover it")
    m = synth.make_mesh(grid)
    got = check(oracle_mod, m, fields(m), section_list(m.nx, m.ny), setting, full=full)
    assert np.count_nonzero(got) > 0


# ---- 3. production widths -------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("setting", [(0, 0.0, False, 23.0, 28.5, 100), (0, 2000.0, False, 32.0, 37.5, 100)], ids=["sigma0", "sigma2000"])
def test_production_widths(sigtrp, oracle_mod, setting):
    """A 1400-column zonal section of an ORCA025 band and a 1000-column meridional section, 75 levels, 100 classes."""
    for m, sec in ((synth.make_mesh("ORCA025", rows=(600, 604)), (20, 1420, 2, 2)), (synth.make_mesh((6, 1021, 75)), (3, 3, 10, 1010))):
        assert npts_of(sec) in (1400, 1000) and m.nz == 75
        got = check(oracle_mod, m, fields(m, boxes=False), [sec, (2, 2, 1, 3)], setting, nk_cases=False)
        assert np.count_nonzero(got[0]) > 10


# ---- 4. missing values, NaN / Inf ------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("setting", [SETTINGS[0], SETTINGS[1], SETTINGS[3]], ids=["sigma0", "sigma2000", "temp"])
def test_missing_values_and_nonfinite(sigtrp, oracle_mod, setting):
    m = synth.make_mesh("SMALL")
    u, v, t, s = fields(m, spval=9999.0)
    j0, i0 = m.ny // 2 - 1, m.nx // 3 - 1
    t[0, j0, 10], t[2, j0 + 1, 15], t[1, j0, 40] = np.nan, np.inf, -np.inf
    t[3, 5, i0], t[0, 9, i0 + 1] = np.nan, np.inf
    assert (u == 9999.0).any() and (v == 9999.0).any() and (s == 9999.0).any()
    check(oracle_mod, m, (u, v, t, s), section_list(m.nx, m.ny), setting, spval=9999.0)


# ---- 5. against the command-line twin ---------------------------------------------------------------------------------------
@gpu
def test_same_as_the_command_line_twin(sigtrp, tmp_path):
    from cdftools_b200 import build
    tools = build.build_host()
    m = synth.make_mesh("SMALL")
    ncfiles.write_mesh(m, tmp_path)
    u = ncfiles.write_gridu(m, tmp_path / "gridU.nc", 1)[0]
    v = ncfiles.write_gridv(m, tmp_path / "gridV.nc", 1)[0]
    t, s = ncfiles.write_gridt(m, tmp_path / "SYN_gridT.nc", 1)[0]
    secs = {"01_zonal": (20, 150, 17, 17), "02_merid": (60, 60, 4, 33), "03_oblique": (10, 20, 5, 9), "04_one": (7, 8, 3, 3),
            "05_lastrow": (1, m.nx, m.ny - 1, m.ny - 1), "06_lastcol": (m.nx - 1, m.nx - 1, 0, m.ny)}
    (tmp_path / "dens_section.dat").write_text("".join(f"{n}\n{' '.join(map(str, b))}\n" for n, b in secs.items()) + "EOF\n")
    r = subprocess.run([tools["cdfsigtrp_gpu"], "-t", "SYN_gridT.nc", "-u", "gridU.nc", "-v", "gridV.nc", "-smin", "23", "-smax", "28.5",
                        "-nbins", "22"], capture_output=True, text=True, cwd=tmp_path, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    twin_nk = [int(x) for x in re.findall(r"(?:NK =|JMM nk)\s+(\d+)", r.stdout)]
    setup(m, list(secs.values()), (0, 0.0, False, 23.0, 28.5, 22))
    got, nk = run_device((u, v, t, s), len(secs), 22)
    kept = [r_ for r_, b in enumerate(secs.values()) if npts_of(b) > 0 and (b[0] == b[1] or b[2] == b[3])]
    assert len(kept) == 5 and twin_nk == [int(nk[r_]) for r_ in kept]
    for r_, name in enumerate(secs):
        if r_ not in kept:
            continue
        f = netcdf_file(str(tmp_path / f"{name}_trpsig.nc"), "r", mmap=False)
        want = f.variables["sigtrp"][0, :, 0, 0].copy()
        f.close()
        assert np.array_equal((got[r_] / 1.e6).astype(f32), want), name


# ---- 6. the device-call contract ---------------------------------------------------------------------------------------------
SETTING = SETTINGS[1]


@pytest.fixture
def small(sigtrp):
    m = synth.make_mesh("ODD")
    secs = section_list(m.nx, m.ny)
    flds = fields(m)
    setup(m, secs, SETTING)
    ref, ref_nk = run_device(flds, len(secs), SETTING[5])
    return m, secs, flds, ref, ref_nk


def outputs(nsec):
    import torch
    return (torch.full((nsec, SETTING[5]), FILL, dtype=torch.float64, device="cuda"),
            torch.full((nsec,), -7, dtype=torch.int32, device="cuda"))


@gpu
def test_inputs_from_the_kernel_just_before(small):
    """The fields are written by a torch kernel on a caller stream right before the call, behind a sleep, with no
    synchronisation in between; a second call on the library's stream follows: both read what was written."""
    import torch
    m, secs, flds, ref, ref_nk = small
    src = [dev(a) for a in flds]
    bufs = [torch.zeros_like(a) for a in src]
    out, nk = outputs(len(secs))
    torch.cuda.synchronize()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        torch.cuda._sleep(20_000_000)
        for b, a in zip(bufs, src):
            b.copy_(a)
        lib.cdfsigtrp_sections_device(*bufs, out, nk, stream=st)
        busy = not st.query()
    torch.cuda.synchronize()
    assert busy
    assert np.array_equal(out.cpu().numpy(), ref, equal_nan=True) and np.array_equal(nk.cpu().numpy(), ref_nk)


@gpu
def test_no_host_device_copies_and_fixed_launches(small):
    """A trace over device calls shows kernels only; every call launches the same four kernels, for 1 section or 30."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    m, secs, flds, ref, _ = small
    d = [dev(a) for a in flds]
    out, nk = outputs(len(secs))
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    n0 = lib.launch_count()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        with torch.cuda.stream(st):
            lib.cdfsigtrp_sections_device(*d, out, nk, stream=st)
            lib.cdfsigtrp_sections_device(*d, out, None, stream=st)
        torch.cuda.synchronize()
    assert lib.launch_count() - n0 == 8
    names = [e.name for e in prof.events()]
    for k in ("sigtrp_sections_prep_kernel", "sigtrp_sections_nk_kernel", "sigtrp_sections_iso_kernel", "sigtrp_sections_bins_kernel"):
        assert any(k in n for n in names), f"{k} not in the trace"
    copies = [n for n in names if "HtoD" in n or "DtoH" in n]
    assert not copies, copies
    assert np.array_equal(out.cpu().numpy(), ref, equal_nan=True)
    deltas = []
    for secs_n in ([secs[0]], [(2 + i, 30 + i % 5, 1 + i % 7, 1 + i % 7) if i % 2 else (3 + i, 3 + i, 1, 2 + i % 7) for i in range(30)]):
        setup(m, secs_n, SETTING)
        o, k = outputs(len(secs_n))
        torch.cuda.synchronize()
        n0 = lib.launch_count()
        lib.cdfsigtrp_sections_device(*d, o, k)
        deltas.append(lib.launch_count() - n0)
        torch.cuda.synchronize()
    assert deltas == [4, 4]


@gpu
def test_repeated_calls_and_a_second_setup(small, oracle_mod):
    """Calls repeat bit for bit; a second setup replaces the plan: the same sections in another list give the same rows."""
    m, secs, flds, ref, ref_nk = small
    again, nk = run_device(flds, len(secs), SETTING[5])
    assert np.array_equal(again, ref, equal_nan=True) and np.array_equal(nk, ref_nk)
    order = [1, 8, 0, 4]
    _, npts = setup(m, [secs[i] for i in order], SETTING)
    assert list(npts) == [npts_of(secs[i]) for i in order]
    got, nk2 = run_device(flds, len(order), SETTING[5])
    assert np.array_equal(got, ref[order], equal_nan=True) and np.array_equal(nk2, ref_nk[order])


def code_of(thunk):
    with pytest.raises(lib.CdfGpuError) as ei:
        thunk()
    return ei.value.code


@gpu
def test_errors(small):
    import torch
    m, secs, flds, _, _ = small
    d = [dev(a) for a in flds]
    out, nk = outputs(len(secs))
    # the wrapper checks tensors before the C call: dtype, element count, device, contiguity
    for bad in ({0: d[0].double()}, {2: d[2][:-1]}, {3: d[3].cpu()}, {1: d[1].transpose(1, 2)}, {4: out[:-1]}, {4: out.float()},
                {5: nk.long()}, {5: nk[:-1]}):
        args = d + [out, nk]
        for i, a in bad.items():
            args[i] = a
        with pytest.raises(ValueError):
            lib.cdfsigtrp_sections_device(*args)
    with pytest.raises(ValueError):
        lib.cdfsigtrp_sections_device(flds[0], *d[1:], out, nk)
    # null pointers straight through the C ABI; a missing U with a meridional section, a missing V with a zonal one
    L, p = lib.load(), [a.data_ptr() for a in d]
    assert L.cdfsigtrp_gpu_sections_device(p[0], p[1], None, p[3], out.data_ptr(), None, None) == ERR_ARG
    assert L.cdfsigtrp_gpu_sections_device(p[0], p[1], p[2], p[3], None, None, None) == ERR_ARG
    assert code_of(lambda: lib.cdfsigtrp_sections_device(None, *d[1:], out, nk)) == ERR_ARG
    assert code_of(lambda: lib.cdfsigtrp_sections_device(d[0], None, *d[2:], out, nk)) == ERR_ARG
    # a plan with only zonal sections takes no U (and one with only meridional sections no V)
    setup(m, [secs[0]], SETTING)
    o1, k1 = outputs(1)
    lib.cdfsigtrp_sections_device(None, *d[1:], o1, k1)
    setup(m, [secs[1]], SETTING)
    lib.cdfsigtrp_sections_device(d[0], None, *d[2:], o1, k1)
    torch.cuda.synchronize()
    # boxes outside the grid, missing mesh arrays, bad mode / nbins
    nx, ny = m.nx, m.ny
    for box in ((1, nx + 1, 3, 3), (0, 5, 3, 3), (2, 9, ny, ny), (2, 9, 0, 0), (nx, nx, 1, 4), (0, 0, 1, 4), (3, 3, 1, ny + 1), (3, 3, -1, 4)):
        assert code_of(lambda: setup(m, [secs[0], box], SETTING)) == ERR_ARG, box
    mode, refdep, teos10, smin, smax, nbins = SETTING

    def mk(sec, full=False, **over):
        kw = {**mesh_arrays(m, full), **over}
        nb, md = kw.pop("nbins", nbins), kw.pop("mode", mode)
        return lambda: lib.cdfsigtrp_sections_setup(np.array([sec]), dsigma_min=smin, dsigma_max=smax, nbins=nb, mode=md, **kw)

    assert code_of(mk(secs[1], e2u=None)) == ERR_ARG
    assert code_of(mk(secs[0], e1v=None)) == ERR_ARG
    assert code_of(mk(secs[0], e3w=None)) == ERR_ARG
    assert code_of(mk(secs[1], e3u=None)) == ERR_ARG
    assert code_of(mk(secs[0], full=True, e3t_1d=None)) == ERR_ARG
    assert code_of(mk(secs[0], mode=3)) == ERR_ARG
    assert code_of(mk(secs[0], nbins=0)) == ERR_ARG
    assert code_of(mk(secs[0], nbins=65535)) == ERR_ARG                     # class limits are a grid dimension
    many = np.tile(np.array([secs[2]]), (65536, 1))                         # so are the sections
    assert code_of(lambda: lib.cdfsigtrp_sections_setup(many, m.gdept_1d, m.gdepw_1d, smin, smax, nbins, e1v=m.e1v, e3t_1d=m.e3t_1d,
                                                        e3w_1d=m.gdepw_1d)) == ERR_ARG
    # before setup
    lib.cdfsigtrp_teardown()
    assert code_of(lambda: lib.cdfsigtrp_sections_device(*d, out, nk)) == ERR_STATE


@gpu
def test_two_devices_refuse(gpu_lib):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    lib.finalize()
    try:
        lib.init_multi(2, "time", 3)
        assert code_of(lambda: lib.cdfsigtrp_sections_device(256, 256, 256, 256, 256, 256)) == ERR_STATE
        assert "one device" in lib.load().cdfgpu_last_error().decode()
        m = synth.make_mesh("ODD")
        assert code_of(lambda: setup(m, [(2, 9, 3, 3)], SETTING)) == ERR_STATE
    finally:
        lib.finalize()
        lib.init(0, 3)


_NO_DEVICE = """
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from cdftools_b200 import lib
for name, call in (("device", lambda: lib.cdfsigtrp_sections_device(256, 256, 256, 256, 256, 256)),
                   ("setup", lambda: lib.cdfsigtrp_sections_setup(np.array([[2, 9, 3, 3]]), np.ones(4, np.float32), np.ones(4, np.float32),
                                                                 24.0, 28.0, 4, e1v=np.ones((5, 12), np.float32), e3t_1d=np.ones(4, np.float32),
                                                                 e3w_1d=np.ones(4, np.float32)))):
    try:
        call()
        sys.exit(name + " succeeded without a device")
    except lib.CdfGpuError as e:
        assert e.code == 5, (name, e.code)   # CDFGPU_ERR_NODEVICE
"""


def test_sections_without_a_device():
    """In a process that sees no device both entry points fail with CDFGPU_ERR_NODEVICE (no CPU fallback)."""
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE, str(ROOT)], capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stdout + r.stderr
