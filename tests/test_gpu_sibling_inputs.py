"""Raw and 16-bit packed records decoded on the device for the sibling tools (cdfgpu_set_sibling_input: the K3 swap and
the K3b unpack of the cdfmoc / cdfmocsig submits, reused by cdfzonal_gpu_*, cdfmhst_gpu_record[_vts] and
cdftransig_gpu_record), and the V-point products of cdfmhst's -v/-t mode formed on the device (mhst_vpoint_kernel).
Every comparison is exact: big-endian float32, host int16 and big-endian int16 records must give what host-order float32
records of the decoded values give, and the command-line twins must write byte-identical files for packed and float
inputs, and for float32 inputs (now decoded on the device) and the same values stored as NC_DOUBLE (decoded on the host)."""
import re
import subprocess

import numpy as np
import pytest
from scipy.io import netcdf_file

from cdftools_b200 import build, ncfiles, synth
from test_gpu_packed import PACK, SP, decoded, quantize
from test_packed_inputs import build_unpack_dump
from util import case_inputs

REPS = ("f32be", "i16", "i16be")      # how a record is handed over, besides host-order float32 ("f32")
NAN = float("nan")


# ---- CPU --------------------------------------------------------------------------------------------------------------
def test_mhst_vpoint_kernel_rounds_every_operation():
    """zvt = fl32(fl32(0.5*fl32(zt+zt')) * zv): two FADD and four FMUL per cell, never an FFMA (one rounding less)."""
    out = subprocess.run(["cuobjdump", "-sass", str(build.build())], capture_output=True, text=True, check=True).stdout
    funcs = re.split(r"\n\s*Function : ", out)
    body = [f for f in funcs if f.startswith("_ZN6cdfgpu18mhst_vpoint_kernel")]
    assert len(body) == 1, "mhst_vpoint_kernel not found in the SASS"
    ops = re.findall(r"\b(FFMA|FADD|FMUL)\b", body[0])
    assert "FFMA" not in ops and ops.count("FADD") >= 2 and ops.count("FMUL") >= 4, ops


# ---- helpers ----------------------------------------------------------------------------------------------------------
def reset_siblings(lib):
    """Every field of every sibling call back to host-order REAL(4), the default."""
    for call, n in ((lib.CALL_ZONAL, 1), (lib.CALL_MHST, 2), (lib.CALL_MHST_VTS, 3), (lib.CALL_TRANSIG, 6)):
        for f in range(n):
            lib.set_sibling_input(call, f, lib.INPUT_F32)


@pytest.fixture
def lib(gpu_lib):
    """The session library; afterwards every sibling field is host-order REAL(4) again, as are the submit fields."""
    yield gpu_lib
    reset_siblings(gpu_lib)
    for f in range(5):
        gpu_lib.set_input_packing(f, gpu_lib.INPUT_F32)
    gpu_lib.set_input_big_endian(False)


def declare(lib, call, field, rep, kind):
    if rep.startswith("f32"):
        lib.set_sibling_input(call, field, lib.INPUT_F32, rep == "f32be")
    else:
        lib.set_sibling_input(call, field, lib.INPUT_I16, rep == "i16be", *PACK[kind], SP)


def handed(raw, kind, rep):
    """The array a caller hands over for the int16 record `raw`: decoded float32 or the int16 values, host order or the
    raw big-endian bytes of the file."""
    a = decoded(raw, kind) if rep.startswith("f32") else raw
    return np.ascontiguousarray(a.byteswap() if rep.endswith("be") else a)


def vpoint(zv, zt, zs):
    """The host loop of cdfmhst's separate-file mode (cdfmhst.f90:313-323), as test_cdfmhst_cli_separate_files states it."""
    zvt, zvs = np.zeros_like(zv), np.zeros_like(zv)
    with np.errstate(over="ignore", invalid="ignore"):   # the non-finite cases are meant
        zvt[:, :-1] = ((np.float32(0.5) * (zt[:, :-1] + zt[:, 1:]).astype(np.float32)).astype(np.float32) * zv[:, :-1]).astype(np.float32)
        zvs[:, :-1] = ((np.float32(0.5) * (zs[:, :-1] + zs[:, 1:]).astype(np.float32)).astype(np.float32) * zv[:, :-1]).astype(np.float32)
    return zvt, zvs


def mhst_setup(lib, m):
    return lib.cdfmhst_setup(m.e1v, m.e3v_0, m.vmask[0].astype(np.float32), m.tmaskatl, m.tmaskpac, m.tmaskind)


def vts_records(m, r):
    v = quantize(synth.make_v_record(m, r), "v", m.vmask == 0)
    t, s = synth.make_ts_record(m, r)
    return v, quantize(t, "t", m.tmask == 0), quantize(s, "s", m.tmask == 0)


# ---- ABI --------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("grid", ["TINY", "ODD", (1442, 12, 6), "2d"])   # 1442: the ORCA025 row; 2d: 333 cells, not 8k
def test_zonal_packed_and_raw_equal_decoded(lib, oracle_mod, grid):
    m = synth.make_mesh("ODD" if grid == "2d" else grid)
    nk = 1 if grid == "2d" else m.nz - 1
    if grid == "2d":
        assert (nk * m.ny * m.nx) % 8 != 0
    msk = m.vmask[:nk].astype(np.float32)
    zm = oracle_mod.zonal_masks(msk[0], m.tmaskatl, m.tmaskind, m.tmaskpac)
    e2 = (m.e1v * np.float32(0.75)).astype(np.float32)
    alpha = (0.5 + np.arange(m.ny) / m.ny).astype(np.float32)
    shape = lib.cdfzonal_setup(m.e1v, e2, zm, msk)
    raws = [quantize(synth.make_v_record(m, r, adversarial=(r == 1))[:nk], "v", m.vmask[:nk] == 0) for r in range(3)]
    for raw in raws:
        ref_sum = lib.cdfzonal_sum(decoded(raw, "v"), shape, alpha)
        ref_mean = lib.cdfzonal_mean(decoded(raw, "v"), shape, 99999.0, True)
        assert np.abs(ref_sum).max() > 0
        for rep in REPS:
            declare(lib, lib.CALL_ZONAL, 0, rep, "v")
            assert np.array_equal(lib.cdfzonal_sum(handed(raw, "v", rep), shape, alpha), ref_sum), rep
            got = lib.cdfzonal_mean(handed(raw, "v", rep), shape, 99999.0, True)
            for a, b in zip(got, ref_mean):
                assert np.array_equal(a, b), rep
            declare(lib, lib.CALL_ZONAL, 0, "f32", "v")
    lib.cdfzonal_teardown()


@pytest.mark.gpu
@pytest.mark.parametrize("zdim", [False, True])
def test_mhst_record_packed_equals_decoded(lib, zdim):
    m = synth.make_mesh("ODD")
    dims = mhst_setup(lib, m)
    land = m.vmask == 0
    for r in range(2):
        v = synth.make_v_record(m, r)
        t, s = synth.make_ts_record(m, r)
        vt, vs = quantize(v * t, "t", land), quantize(v * s, "s", land)
        reset_siblings(lib)
        ref = lib.cdfmhst_record(decoded(vt, "t"), decoded(vs, "s"), dims, zdim)
        for rep_t, rep_s in (("i16", "i16be"), ("i16be", "f32be"), ("f32be", "i16")):
            declare(lib, lib.CALL_MHST, 0, rep_t, "t")
            declare(lib, lib.CALL_MHST, 1, rep_s, "s")
            got = lib.cdfmhst_record(handed(vt, "t", rep_t), handed(vs, "s", rep_s), dims, zdim)
            assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), (rep_t, rep_s)
    lib.cdfmhst_teardown()


@pytest.mark.gpu
@pytest.mark.parametrize("zdim", [False, True])
def test_mhst_record_vts_equals_host_products(lib, zdim):
    """cdfmhst_gpu_record_vts on V, T, S = cdfmhst_gpu_record on the products the host loop forms, including NaN and Inf
    cells (which pin the fp32 order), and for packed and raw V / T / S."""
    m = synth.make_mesh("SMALL")
    dims = mhst_setup(lib, m)
    for r in range(2):
        v, t, s = vts_records(m, r)
        zv, zt, zs = decoded(v, "v"), decoded(t, "t"), decoded(s, "s")
        if r == 1:   # non-finite cells, and sums that overflow fp32
            zt[2, 5, 7], zt[3, 6, 9], zs[1, 4, 11], zv[4, 8, 12] = NAN, np.inf, -np.inf, np.inf
            zt[0, 10, 20], zt[0, 11, 20] = np.float32(3e38), np.float32(3e38)
        reset_siblings(lib)
        ref = lib.cdfmhst_record(*vpoint(zv, zt, zs), dims, zdim)
        got = lib.cdfmhst_record_vts(zv, zt, zs, dims, zdim)
        assert np.array_equal(got[0], ref[0], equal_nan=True) and np.array_equal(got[1], ref[1], equal_nan=True)
        if r == 1:
            assert np.isnan(ref[0]).any()
            for f in range(3):
                declare(lib, lib.CALL_MHST_VTS, f, "f32be", "v")
            got = lib.cdfmhst_record_vts(zv.byteswap(), zt.byteswap(), zs.byteswap(), dims, zdim)
            assert np.array_equal(got[0], ref[0], equal_nan=True) and np.array_equal(got[1], ref[1], equal_nan=True)
            continue
        for reps in (("i16", "i16", "i16"), ("i16be", "f32be", "i16be"), ("f32", "i16be", "i16")):
            for f, (rep, kind) in enumerate(zip(reps, ("v", "t", "s"))):
                declare(lib, lib.CALL_MHST_VTS, f, rep, kind)
            got = lib.cdfmhst_record_vts(handed(v, "v", reps[0]), handed(t, "t", reps[1]), handed(s, "s", reps[2]), dims, zdim)
            assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), reps
    lib.cdfmhst_teardown()


def transig_frames(m, n):
    land_u, land_v, land_t = m.umask[:-1] == 0, m.vmask[:-1] == 0, m.tmask[:-1] == 0
    out = []
    for r in range(n):
        t, s = (x[:-1] for x in synth.make_ts_record(m, r))
        e3 = [quantize((m.e3v_0[:-1] * np.float32(f + 0.01 * r)).astype(np.float32), "e3", np.zeros(land_v.shape, bool))
              for f in (1.01, 1.0)]
        for e in e3:
            e[e == 32767] = 100   # physical thicknesses
        out.append([quantize((synth.make_v_record(m, 500 + r) * m.umask)[:-1], "v", land_u),
                    quantize(synth.make_v_record(m, r)[:-1], "v", land_v), quantize(t, "t", land_t), quantize(s, "s", land_t)] + e3)
    return out


TRANSIG_KINDS = ("v", "v", "t", "s", "e3", "e3")


@pytest.mark.gpu
@pytest.mark.parametrize("vvl", [False, True])
def test_transig_mixed_kinds_accumulate_bit_identical(lib, vvl):
    m = synth.make_mesh("SMALL")
    pref, nb, smin, scal, zoom, smn = lib.TRANSIG_CODES["1000"]
    _, _, itab, step = lib.transig_bins(nb, smin, scal, zoom, smn)
    e2u = (m.e1u * np.float32(0.9)).astype(np.float32)
    frames = transig_frames(m, 5)
    nf = 6 if vvl else 4
    lperio = bool(m.glamv[0, 0] == m.glamv[0, m.nx - 2])

    def run(reps_of, flag=False):
        e3 = (None, None) if vvl else (decoded(frames[0][4], "e3"), decoded(frames[0][5], "e3"))
        shape = lib.cdftransig_setup(e2u, m.e1v, *e3, m.nz, nb, pref, smin, step, itab, lperio=lperio)
        lib.set_input_big_endian(flag)
        for r, fr in enumerate(frames):
            reps = reps_of(r)
            for a in range(6):
                declare(lib, lib.CALL_TRANSIG, a, reps[a], TRANSIG_KINDS[a])
            arg = [handed(fr[a], TRANSIG_KINDS[a], reps[a]) for a in range(nf)]
            if flag:   # the process-wide flag swaps every field on top of its declaration
                arg = [np.ascontiguousarray(x.byteswap()) for x in arg]
            lib.cdftransig_record(*arg[:4], set_masks=r < 3, e3u_vvl=arg[4] if vvl else None, e3v_vvl=arg[5] if vvl else None)
        out = lib.cdftransig_fetch(shape)
        lib.set_input_big_endian(False)
        lib.cdftransig_teardown()
        return out

    ref = run(lambda r: ("f32",) * 6)
    assert np.abs(ref[0]).max() > 0 and np.abs(ref[1]).max() > 0
    all_reps = ("f32",) + REPS
    got = run(lambda r: tuple(all_reps[(r + a) % 4] for a in range(6)))
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])
    # cdfgpu_set_input_big_endian with undeclared fields still swaps them all; a host-order declaration is swapped too
    legacy = run(lambda r: ("f32",) * 6 if r % 2 == 0 else ("i16", "f32", "i16", "f32", "i16", "f32"), flag=True)
    assert np.array_equal(legacy[0], ref[0]) and np.array_equal(legacy[1], ref[1])


@pytest.mark.gpu
def test_zonal_and_mhst_ignore_the_process_byte_order_and_packings_are_independent(lib, oracle_mod):
    m = synth.make_mesh("TINY")
    nk = m.nz - 1
    msk = m.vmask[:nk].astype(np.float32)
    zv = decoded(quantize(synth.make_v_record(m, 0)[:nk], "v", m.vmask[:nk] == 0), "v")
    shape = lib.cdfzonal_setup(m.e1v, m.e1v, oracle_mod.zonal_masks(msk[0]), msk)
    dims = mhst_setup(lib, m)
    v, t, s = (decoded(a, k) for a, k in zip(vts_records(m, 0), ("v", "t", "s")))
    ib, e3m = case_inputs(oracle_mod, m, synth)
    moc_shape = lib.cdfmoc_setup(m.e1v, e3m, ib)

    def siblings():
        return [lib.cdfzonal_sum(zv, shape), lib.cdfzonal_mean(zv, shape, 0.0, True)[0], *lib.cdfmhst_record(v * t, v * s, dims),
                *lib.cdfmhst_record_vts(v, t, s, dims)]

    def moc():
        lib.cdfmoc_submit(0, 0, v[:-1])
        return lib.cdfmoc_fetch(0, np.empty(moc_shape))

    ref, ref_moc = siblings(), moc()
    lib.set_input_big_endian(True)       # the submit calls would now swap; the zonal / mhst calls do not look
    got = siblings()
    lib.set_input_big_endian(False)
    assert all(np.array_equal(a, b) for a, b in zip(got, ref))
    for f in range(5):
        lib.set_input_packing(f, lib.INPUT_I16, 1e-4, 0.0, SP)   # the submit fields say int16 ...
    got = siblings()                                             # ... the sibling calls still read float32
    for f in range(5):
        lib.set_input_packing(f, lib.INPUT_F32)
    assert all(np.array_equal(a, b) for a, b in zip(got, ref))
    for call, n in ((lib.CALL_ZONAL, 1), (lib.CALL_MHST, 2), (lib.CALL_MHST_VTS, 3), (lib.CALL_TRANSIG, 6)):
        for f in range(n):
            lib.set_sibling_input(call, f, lib.INPUT_I16, True, 1e-4, 0.0, SP)   # the sibling fields say int16 ...
    assert np.array_equal(moc(), ref_moc)                                        # ... cdfmoc still reads float32
    lib.cdfzonal_teardown()
    lib.cdfmhst_teardown()
    lib.cdfmoc_teardown()


@pytest.mark.gpu
def test_set_sibling_input_rejects_bad_arguments(lib):
    bad = [(4, 0, 0), (-1, 0, 0), (0, 1, 0), (1, 2, 0), (2, 3, 0), (3, 6, 0), (3, -1, 0), (0, 0, 2), (0, 0, -1),
           (0, 0, 1, False, NAN), (3, 5, 1, True, 1.0, float("inf"))]
    for args in bad:
        with pytest.raises(lib.CdfGpuError) as e:
            lib.set_sibling_input(*args)
        assert e.value.code == 2, args   # CDFGPU_ERR_ARG
    lib.set_sibling_input(3, 5, lib.INPUT_F32, True, NAN)   # REAL(4) takes no unpacking constants


# ---- command-line twins -----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tools():
    return build.build_host()


def write_nc(path, m, zdim, nrec, fields):
    """fields = {name: (records, {attribute: value})}: records (nz,ny,nx) or (ny,nx), int16 / float32 / float64."""
    nz, ny, nx = m.e3v_0.shape
    f = netcdf_file(str(path), "w", version=2)
    f.createDimension("time_counter", None)
    f.createDimension("x", nx)
    f.createDimension("y", ny)
    f.createDimension(zdim, nz)
    f.start_date = np.int32(20260101)
    f.CONFIG = "SYN"
    tc = f.createVariable("time_counter", "d", ("time_counter",))
    tc.units = "seconds since 2026-01-01 00:00:00"
    for name, (recs, atts) in fields.items():
        dims = ("time_counter",) + ((zdim,) if recs[0].ndim == 3 else ()) + ("y", "x")
        v = f.createVariable(name, {np.int16: "h", np.float32: "f", np.float64: "d"}[recs[0].dtype.type], dims)
        for k, a in atts.items():
            setattr(v, k, a)
        for r in range(nrec):
            v[r] = recs[r]
    for r in range(nrec):
        tc[r] = 432000.0 * (r + 0.5)
    f.close()


def stored(raws, kind, how, missing="missing_value"):
    """The records and attributes of one variable: packed int16, or the decoded values as float32 / float64."""
    if how == "packed":
        sf, ao = PACK[kind]
        return raws, {"scale_factor": np.float32(sf), "add_offset": np.float32(ao), missing: np.int16(SP)}
    dt = np.float32 if how == "float" else np.float64
    return [decoded(a, kind).astype(dt) for a in raws], {missing: dt(SP)}


def run_cli(tool, args, cwd):
    r = subprocess.run([str(tool)] + args, capture_output=True, text=True, cwd=cwd, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


def outputs(d, names):
    return {n: (d / n).read_bytes() for n in names}


def case_dirs(tmp_path, m, hows):
    for how in hows:
        ncfiles.write_mesh(m, tmp_path / how)
    return {how: tmp_path / how for how in hows}


HOWS = ("packed", "float", "double")


@pytest.mark.gpu
def test_cli_zonal_packed_float_and_double_inputs_agree(tools, tmp_path):
    m = synth.make_mesh("ORCA2")
    nrec = 2
    v3 = [quantize(synth.make_v_record(m, r), "v", m.vmask == 0) for r in range(nrec)]
    v2 = [quantize(synth.make_ts_record(m, r)[0][0], "t", m.tmask[0] == 0) for r in range(nrec)]   # 2-D, packed
    d = case_dirs(tmp_path, m, HOWS)
    for how in HOWS:
        write_nc(d[how] / "in.nc", m, "depthv", nrec, {"vomecrty": stored(v3, "v", how), "sosstsst": stored(v2, "t", how)})
    cases = [("cdfzonalsum_gpu", ["-f", "in.nc", "-p", "V", "-b", "new_maskglo.nc"], ["zonalsum.nc"]),
             ("cdfzonalmean_gpu", ["-f", "in.nc", "-p", "V", "-b", "new_maskglo.nc", "-max"], ["zonalmean.nc"])]
    for tool, args, outs in cases:
        res = {}
        for how in HOWS:
            run_cli(tools[tool], args, d[how])
            res[how] = outputs(d[how], outs)
        assert res["packed"] == res["float"], tool
        assert res["float"] == res["double"], tool   # device decode of float32 = host decode of NC_DOUBLE


@pytest.mark.gpu
def test_cli_zonal_savelog10_and_mixed_fields(tools, tmp_path):
    """A savelog10 field stays on the host decode (glibc powf) next to a packed field decoded on the device."""
    dump = build_unpack_dump(tmp_path)
    m = synth.make_mesh("TINY")
    nrec = 2
    v3 = [quantize(synth.make_v_record(m, r), "v", m.vmask == 0) for r in range(nrec)]
    lg = [quantize(synth.make_ts_record(m, r)[0], "t", m.tmask == 0) for r in range(nrec)]
    d = case_dirs(tmp_path, m, ("log", "float"))
    sf, ao = PACK["t"]
    write_nc(d["log"] / "in.nc", m, "depthv", nrec, {"vomecrty": stored(v3, "v", "packed"), "votemper": (lg, {
        "scale_factor": np.float32(sf * 1e-3), "add_offset": np.float32(ao * 1e-2), "missing_value": np.int16(SP),
        "savelog10": np.int32(1)})})
    vals, info = dump(d["log"] / "in.nc", "votemper")
    assert not info["packed"]
    vals = vals.reshape((nrec,) + m.e3v_0.shape)
    write_nc(d["float"] / "in.nc", m, "depthv", nrec, {"vomecrty": stored(v3, "v", "float"),
                                                        "votemper": ([vals[r] for r in range(nrec)], {"missing_value": np.float32(SP)})})
    for how in ("log", "float"):
        run_cli(tools["cdfzonalsum_gpu"], ["-f", "in.nc", "-p", "V"], d[how])
    assert (d["log"] / "zonalsum.nc").read_bytes() == (d["float"] / "zonalsum.nc").read_bytes()


MHST_OUTS = ["mhst.nc", "zonal_heat_trp.dat", "zonal_salt_trp.dat"]


@pytest.mark.gpu
def test_cli_mhst_vt_file(tools, tmp_path):
    m = synth.make_mesh("ODD")
    nrec = 2
    land = m.vmask == 0
    vt, vs = [], []
    for r in range(nrec):
        v = synth.make_v_record(m, r)
        t, s = synth.make_ts_record(m, r)
        vt.append(quantize(v * t, "t", land))
        vs.append(quantize(v * s, "s", land))
    d = case_dirs(tmp_path, m, HOWS)
    for how in HOWS:
        write_nc(d[how] / "VT.nc", m, "depthv", nrec, {"vomevt": stored(vt, "t", how), "vomevs": stored(vs, "s", how)})
        run_cli(tools["cdfmhst_gpu"], ["-vt", "VT.nc", "-MST", "-Zdim"], d[how])
    res = {how: outputs(d[how], MHST_OUTS) for how in HOWS}
    assert res["packed"] == res["float"] and res["float"] == res["double"]


@pytest.mark.gpu
def test_cli_mhst_separate_files(tools, tmp_path):
    """-v -t -s: packed, float, double and mixed files give the same outputs, and the variables equal those of -vt mode on a
    VT file holding the products the host loop forms."""
    m = synth.make_mesh("SMALL")
    nrec = 2
    recs = [vts_records(m, r) for r in range(nrec)]
    hows = HOWS + ("mixed", "vt")
    d = case_dirs(tmp_path, m, hows)
    for how in HOWS + ("mixed",):
        hv, ht, hs = (how,) * 3 if how != "mixed" else ("packed", "float", "packed")
        write_nc(d[how] / "gridV.nc", m, "depthv", nrec, {"vomecrty": stored([r[0] for r in recs], "v", hv)})
        write_nc(d[how] / "gridT.nc", m, "deptht", nrec, {"votemper": stored([r[1] for r in recs], "t", ht, "_FillValue")})
        write_nc(d[how] / "gridS.nc", m, "deptht", nrec, {"vosaline": stored([r[2] for r in recs], "s", hs, "_FillValue")})
        run_cli(tools["cdfmhst_gpu"], ["-v", "gridV.nc", "-t", "gridT.nc", "-s", "gridS.nc", "-MST"], d[how])
    res = {how: outputs(d[how], MHST_OUTS) for how in HOWS + ("mixed",)}
    assert res["packed"] == res["float"] and res["float"] == res["double"] and res["mixed"] == res["float"]
    prods = [vpoint(decoded(v, "v"), decoded(t, "t"), decoded(s, "s")) for v, t, s in recs]
    write_nc(d["vt"] / "VT.nc", m, "depthv", nrec, {"vomevt": ([p[0] for p in prods], {}), "vomevs": ([p[1] for p in prods], {})})
    run_cli(tools["cdfmhst_gpu"], ["-vt", "VT.nc", "-MST"], d["vt"])
    a = netcdf_file(str(d["float"] / "mhst.nc"), "r", mmap=False)
    b = netcdf_file(str(d["vt"] / "mhst.nc"), "r", mmap=False)
    names = [n for n in a.variables if n.startswith(("zomht", "zomst"))]
    assert len(names) == 12
    for n in names:
        assert np.array_equal(a.variables[n][:], b.variables[n][:]), n
    a.close()
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("vvl", [False, True])
def test_cli_transig(tools, tmp_path, vvl):
    m = synth.make_mesh("SMALL")
    frames = transig_frames(m, 4)
    full = lambda a: np.concatenate([a, a[-1:]])   # the files hold nz levels; the bottom one is not read
    hows = HOWS + ("mixed",)
    d = case_dirs(tmp_path, m, hows)
    for how in hows:
        hu = how if how != "mixed" else "packed"
        hf = how if how != "mixed" else "float"
        for t, tag in enumerate(("y2026m01", "y2026m02")):
            fr = frames[2 * t:2 * t + 2]
            pre = d[how] / f"SYN-B200_{tag}_grid"
            fu = {"vozocrtx": stored([full(f[0]) for f in fr], "v", hu)}
            fv = {"vomecrty": stored([full(f[1]) for f in fr], "v", hf)}
            if vvl:
                fu["e3u"] = stored([full(f[4]) for f in fr], "e3", hf)
                fv["e3v"] = stored([full(f[5]) for f in fr], "e3", hu)
            write_nc(str(pre) + "U.nc", m, "depthu", 2, fu)
            write_nc(str(pre) + "V.nc", m, "depthv", 2, fv)
            write_nc(str(pre) + "T.nc", m, "deptht", 2, {"votemper": stored([full(f[2]) for f in fr], "t", hu, "_FillValue")})
            write_nc(str(pre) + "S.nc", m, "deptht", 2, {"vosaline": stored([full(f[3]) for f in fr], "s", hf, "_FillValue")})
        run_cli(tools["cdftransig_xy3d_gpu"], ["-c", "SYN-B200", "-l", "y2026m01", "y2026m02", "-S", "-o", "uv.nc"]
                + (["-vvl"] if vvl else []), d[how])
    res = {how: (d[how] / "uv.nc").read_bytes() for how in hows}
    assert res["packed"] == res["float"] == res["double"] == res["mixed"]
    f = netcdf_file(str(d["float"] / "uv.nc"), "r", mmap=False)
    assert np.abs(f.variables["vovxysig"][:]).max() > 0
    f.close()
