"""16-bit packed records unpacked on the device (K3b, cdfgpu_set_input_packing): handing the library the int16 values of
a packed record must give BIT-IDENTICAL results to handing it the float32 values getvar would have produced (the NumPy
restatement of test_packed_inputs.py, itself checked against the host reader).  Through the ABI (cdfmoc, cdfmocsig with
-eiv / -vvl and mixed fields, -decomp, big-endian raw bytes, several slots in flight, two devices) and through the
command-line twins (packed files give the same output files, byte for byte, as float files holding the decoded values)."""
import os
import subprocess

import numpy as np
import pytest
from scipy.io import netcdf_file

from cdftools_b200 import build, synth
from test_packed_inputs import build_unpack_dump, unpack_i16
from util import case_inputs

pytestmark = pytest.mark.gpu

SP = -32768                                  # the missing value of the packed fields
PACK = {"v": (1.0e-4, 0.0), "t": (1.0e-3, 15.0), "s": (5.0e-4, 35.0), "eiv": (2.0e-6, 0.0), "e3": (1.0e-2, 250.0)}


@pytest.fixture
def lib(gpu_lib):
    """The session library, with every field back to REAL(4) and host byte order afterwards."""
    yield gpu_lib
    for f in range(5):
        gpu_lib.set_input_packing(f, gpu_lib.INPUT_F32)
    gpu_lib.set_input_big_endian(False)


def quantize(x, kind, land):
    """int16 record whose unpacking approximates x; land cells hold the missing value, a few cells the extremes."""
    sf, ao = PACK[kind]
    raw = np.clip(np.rint((x.astype(np.float64) - ao) / sf), -32767, 32767).astype(np.int16)
    raw[land] = SP
    flat = raw.reshape(-1)
    flat[7::997] = 32767
    flat[11::1009] = -32767
    return raw


def decoded(raw, kind):
    return unpack_i16(raw, *PACK[kind], SP)


def declare(lib, field, kind):
    lib.set_input_packing(field, lib.INPUT_I16, *PACK[kind], SP)


def hand(a, big_endian):
    """What the caller hands over: host order, or the raw big-endian bytes of the file."""
    return np.ascontiguousarray(a.byteswap() if big_endian else a)


def v_records(m, n):
    land = (m.vmask[:-1] == 0)
    return [quantize(synth.make_v_record(m, r, adversarial=(r % 2 == 1))[:-1], "v", land) for r in range(n)]


def ts_records(m, n):
    land = (m.tmask[:-1] == 0)
    out = []
    for r in range(n):
        t, s = (x[:-1] for x in synth.make_ts_record(m, r))
        out.append((quantize(t, "t", land), quantize(s, "s", land)))
    return out


# ---- ABI --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("big_endian", [False, True])
@pytest.mark.parametrize("grid", ["TINY", "ODD", (1442, 12, 6)])   # (1442, ., .): the ORCA025 row width
def test_cdfmoc_packed_equals_decoded(lib, oracle_mod, grid, big_endian):
    m = synth.make_mesh(grid)
    ib, e3m = case_inputs(oracle_mod, m, synth)
    nz, ny, nb = lib.cdfmoc_setup(m.e1v, e3m, ib)
    raws = v_records(m, 5)
    ns = 3

    def run(records):   # several slots in flight
        out = np.empty((len(records), nz, ny, nb))
        for r0 in range(0, len(records), ns):
            idx = range(r0, min(len(records), r0 + ns))
            for r in idx:
                lib.cdfmoc_submit(r % ns, r, records[r])
            for r in idx:
                lib.cdfmoc_fetch(r % ns, out[r])
        return out

    ref = run([decoded(a, "v") for a in raws])
    declare(lib, 0, "v")
    lib.set_input_big_endian(big_endian)
    pins = []
    for a in raws:   # page-locked int16 buffers, as a host reading the file would use
        p = lib.PinnedArray(a.shape, np.int16)
        p.array[...] = hand(a, big_endian)
        pins.append(p)
    try:
        got = run([p.array for p in pins])
    finally:
        for p in pins:
            p.free()
    assert np.array_equal(got, ref)
    lib.cdfmoc_teardown()


@pytest.mark.parametrize("big_endian", [False, True])
@pytest.mark.parametrize("config", ["all_packed", "mixed_vvl"])
def test_cdfmocsig_packed_equals_decoded(lib, config, big_endian):
    m = synth.make_mesh("SMALL")
    ib = synth.setup_masks(m)
    vvl = config == "mixed_vvl"
    nrec = 4
    vs, ts = v_records(m, nrec), ts_records(m, nrec)
    eivs = [quantize((0.01 * synth.make_v_record(m, 1000 + r)).astype(np.float32)[:-1], "eiv", m.vmask[:-1] == 0) for r in range(nrec)]
    e3s = [quantize((m.e3v_0[:-1] * np.float32(1.0 + 0.01 * r)).astype(np.float32), "e3", np.zeros(m.e3v_0[:-1].shape, bool))
           for r in range(nrec)]
    for e in e3s:
        e[e == 32767] = 100   # keep the layer thicknesses physical (no missing value in e3v)
    # field -> (records, kind); the mixed configuration leaves zt and zveiv as REAL(4)
    fields = {0: (vs, "v"), 1: ([t for t, _ in ts], "t"), 2: ([s for _, s in ts], "s"), 3: (eivs, "eiv")}
    if vvl:
        fields[4] = (e3s, "e3")
    packed = {0, 1, 2, 3} if not vvl else {0, 2, 4}
    lib.cdfmocsig_setup(m.e1v, None if vvl else m.e3v_0, ib, m.nz, 158, 30.0, 0.05, 2000.0, lib.EOS80, float(SP), float(SP), float(SP))
    ns = 3

    def run(pack):
        for f in range(5):
            if f in pack:
                declare(lib, f, fields[f][1])
            else:
                lib.set_input_packing(f, lib.INPUT_F32)
        lib.set_input_big_endian(big_endian if pack else False)
        out = np.empty((nrec, m.ny, 158, 5))
        for r0 in range(0, nrec, ns):
            idx = range(r0, min(nrec, r0 + ns))
            for r in idx:
                arg = [None] * 5
                for f, (recs, kind) in fields.items():
                    a = recs[r] if f in pack else decoded(recs[r], kind)
                    arg[f] = hand(a, big_endian) if pack else a
                lib.cdfmocsig_submit(r % ns, r, *arg)
            for r in idx:
                lib.cdfmocsig_fetch(r % ns, out[r])
        return out

    ref = run(set())
    got = run(packed)
    assert np.abs(ref).max() > 0
    assert np.array_equal(got, ref)
    lib.cdfmocsig_teardown()


@pytest.mark.parametrize("big_endian", [False, True])
def test_cdfmoc_decomp_packed_equals_decoded(lib, oracle_mod, big_endian):
    m = synth.make_mesh("SMALL")
    ib, e3m = case_inputs(oracle_mod, m, synth)
    shape = lib.cdfmoc_setup(m.e1v, e3m, ib)
    lib.cdfmoc_decomp_setup(m.e1u, m.gphiv, m.gdept_1d, m.umask.astype(np.int16), m.tmask.astype(np.int16))
    vs, ts = v_records(m, 2), ts_records(m, 2)
    ref = []
    for r in range(2):
        lib.cdfmoc_decomp_submit(0, r, decoded(vs[r], "v"), decoded(ts[r][0], "t"), decoded(ts[r][1], "s"))
        ref.append(lib.cdfmoc_decomp_fetch(0, shape))
    for f, kind in enumerate(("v", "t", "s")):
        declare(lib, f, kind)
    lib.set_input_big_endian(big_endian)
    for r in range(2):
        lib.cdfmoc_decomp_submit(0, r, hand(vs[r], big_endian), hand(ts[r][0], big_endian), hand(ts[r][1], big_endian))
        got = lib.cdfmoc_decomp_fetch(0, shape)
        for k in ("total", "sh", "bt", "ag"):
            assert np.array_equal(got[k], ref[r][k]), (r, k)
    lib.cdfmoc_teardown()


def test_set_input_packing_rejects_bad_arguments(lib):
    for args in [(5, 1), (-1, 0), (0, 2), (0, -1), (0, 1, float("nan")), (0, 1, 1.0, float("inf"))]:
        with pytest.raises(lib.CdfGpuError) as e:
            lib.set_input_packing(*args)
        assert e.value.code == 2, args   # CDFGPU_ERR_ARG
    lib.set_input_packing(4, lib.INPUT_F32, float("nan"))   # REAL(4) takes no unpacking constants


@pytest.mark.parametrize("shard", ["time", "lat"])
def test_packed_two_devices_equal_one(lib, shard):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    m = synth.make_mesh("ORCA2")
    ib = synth.setup_masks(m)
    e3m = synth.setup_e3v_masked(m)
    nrec = 6
    vs, ts = v_records(m, nrec), ts_records(m, nrec)
    for f, kind in enumerate(("v", "t", "s")):
        declare(lib, f, kind)
    lib.set_input_big_endian(True)

    def run_all():
        ns = lib.nslots()
        nz, ny, nb = lib.cdfmoc_setup(m.e1v, e3m, ib)
        moc = np.empty((nrec, nz, ny, nb))
        sig = np.empty((nrec, m.ny, 158, 5))
        for r0 in range(0, nrec, ns):
            for r in range(r0, min(nrec, r0 + ns)):
                lib.cdfmoc_submit(r % ns, r, hand(vs[r], True))
            for r in range(r0, min(nrec, r0 + ns)):
                lib.cdfmoc_fetch(r % ns, moc[r])
        lib.cdfmocsig_setup(m.e1v, m.e3v_0, ib, m.nz, 158, 30.0, 0.05, 2000.0, lib.EOS80, float(SP), float(SP), float(SP))
        for r0 in range(0, nrec, ns):
            for r in range(r0, min(nrec, r0 + ns)):
                lib.cdfmocsig_submit(r % ns, r, hand(vs[r], True), hand(ts[r][0], True), hand(ts[r][1], True))
            for r in range(r0, min(nrec, r0 + ns)):
                lib.cdfmocsig_fetch(r % ns, sig[r])
        lib.cdfmoc_teardown()
        lib.cdfmocsig_teardown()
        return moc, sig

    one = run_all()
    lib.finalize()
    try:
        lib.init_multi(2, shard, 3)
        lib.set_input_big_endian(True)
        two = run_all()
    finally:
        lib.finalize()
        lib.init(0, 3)
    assert np.array_equal(one[0], two[0]) and np.array_equal(one[1], two[1])


# ---- command-line twins -----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tools():
    return build.build_host()


def write_records(path, m, zdim, nrec, fields):
    """A gridV / gridT style file: fields = {name: (records (nz-1, ny, nx) int16 or float32, {attribute: value})}; the
    bottom level, which no tool reads, is written as the missing value."""
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
        v = f.createVariable(name, "h" if recs[0].dtype == np.int16 else "f", ("time_counter", zdim, "y", "x"))
        for k, a in atts.items():
            setattr(v, k, a)
        for r in range(nrec):
            full = np.full((nz, ny, nx), SP, recs[r].dtype)
            full[:-1] = recs[r]
            v[r] = full
    for r in range(nrec):
        tc[r] = 432000.0 * (r + 0.5)
    f.close()


def packed_and_float(m, tmp, kinds, nrec, zdim, recs, missing="missing_value"):
    """Writes tmp/packed/<file> with the int16 records and tmp/float/<file> with their decoded values."""
    for sub in ("packed", "float"):
        (tmp / sub).mkdir(exist_ok=True)
    fname = "gridV.nc" if zdim == "depthv" else "gridT.nc"
    pk, fl = {}, {}
    for name, kind in kinds.items():
        sf, ao = PACK[kind]
        pk[name] = (recs[name], {"scale_factor": np.float32(sf), "add_offset": np.float32(ao), missing: np.int16(SP)})
        fl[name] = ([decoded(a, kind) for a in recs[name]], {missing: np.float32(SP)})
    write_records(tmp / "packed" / fname, m, zdim, nrec, pk)
    write_records(tmp / "float" / fname, m, zdim, nrec, fl)


def _run(tool, args, cwd, env=None):
    r = subprocess.run([tool] + args, capture_output=True, text=True, cwd=cwd, timeout=600, env=dict(os.environ, **(env or {})))
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


def test_cli_packed_files_give_identical_outputs(tools, tmp_path):
    from cdftools_b200 import ncfiles
    m = synth.make_mesh("SMALL")
    nrec = 4
    vs, ts = v_records(m, nrec), ts_records(m, nrec)
    eivs = [quantize((0.01 * synth.make_v_record(m, 1000 + r)).astype(np.float32)[:-1], "eiv", m.vmask[:-1] == 0) for r in range(nrec)]
    packed_and_float(m, tmp_path, {"vomecrty": "v", "vomeeivv": "eiv"}, nrec, "depthv", {"vomecrty": vs, "vomeeivv": eivs})
    packed_and_float(m, tmp_path, {"votemper": "t", "vosaline": "s"}, nrec, "deptht",
                     {"votemper": [t for t, _ in ts], "vosaline": [s for _, s in ts]}, missing="_FillValue")
    cases = [("cdfmoc_gpu", ["-v", "gridV.nc"], "moc.nc"),
             ("cdfmoc_gpu", ["-v", "gridV.nc", "-t", "gridT.nc", "-decomp"], "moc.nc"),
             ("cdfmocsig_gpu", ["-v", "gridV.nc", "-t", "gridT.nc", "-r", "2000", "-eiv"], "mocsig.nc"),
             ("cdfmocsig_gpu", ["-v", "gridV.nc", "-t", "gridT.nc", "-r", "0", "-isodep"], "mocsig.nc")]
    for sub in ("packed", "float"):
        ncfiles.write_mesh(m, tmp_path / sub)
    for tool, args, out in cases:
        res = {}
        for sub in ("packed", "float"):
            _run(tools[tool], args, tmp_path / sub)
            res[sub] = (tmp_path / sub / out).read_bytes()
        assert res["packed"] == res["float"], f"{tool} {' '.join(args)}: packed input gives a different {out}"
    # a mix of a packed and a float32 field in one record (T packed, S float)
    ncfiles.write_mesh(m, tmp_path / "mix")
    (tmp_path / "mix" / "gridV.nc").write_bytes((tmp_path / "packed" / "gridV.nc").read_bytes())
    write_records(tmp_path / "mix" / "gridT.nc", m, "deptht", nrec,
                  {"votemper": ([t for t, _ in ts], {"scale_factor": np.float32(PACK["t"][0]), "add_offset": np.float32(PACK["t"][1]),
                                                     "_FillValue": np.int16(SP)}),
                   "vosaline": ([decoded(s, "s") for _, s in ts], {"_FillValue": np.float32(SP)})})
    _run(tools["cdfmocsig_gpu"], ["-v", "gridV.nc", "-t", "gridT.nc", "-r", "2000", "-eiv"], tmp_path / "mix")
    _run(tools["cdfmocsig_gpu"], ["-v", "gridV.nc", "-t", "gridT.nc", "-r", "2000", "-eiv"], tmp_path / "float")
    assert (tmp_path / "mix" / "mocsig.nc").read_bytes() == (tmp_path / "float" / "mocsig.nc").read_bytes()


@pytest.mark.parametrize("shard", ["time", "lat"])
def test_cli_packed_two_devices(tools, tmp_path, shard):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from cdftools_b200 import ncfiles
    m = synth.make_mesh("ORCA2")
    nrec = 5
    vs, ts = v_records(m, nrec), ts_records(m, nrec)
    packed_and_float(m, tmp_path, {"vomecrty": "v"}, nrec, "depthv", {"vomecrty": vs})
    packed_and_float(m, tmp_path, {"votemper": "t", "vosaline": "s"}, nrec, "deptht",
                     {"votemper": [t for t, _ in ts], "vosaline": [s for _, s in ts]})
    d = tmp_path / "packed"
    ncfiles.write_mesh(m, d)
    for tool, args in (("cdfmoc_gpu", ["-v", "gridV.nc"]), ("cdfmocsig_gpu", ["-v", "gridV.nc", "-t", "gridT.nc", "-r", "2000"])):
        _run(tools[tool], args + ["-o", "one.nc"], d, {"CDFGPU_DEVICES": "1"})
        _run(tools[tool], args + ["-o", "two.nc"], d, {"CDFGPU_DEVICES": "2", "CDFGPU_SHARD": shard})
        assert (d / "one.nc").read_bytes() == (d / "two.nc").read_bytes(), (tool, shard)


def test_cli_savelog10_keeps_the_host_decode(tools, tmp_path):
    """savelog10 is applied on the host (glibc powf): the output equals that of a float file holding what read_f32 gives."""
    from cdftools_b200 import ncfiles
    dump = build_unpack_dump(tmp_path)
    m = synth.make_mesh("TINY")
    nrec = 2
    vs = v_records(m, nrec)
    (tmp_path / "log").mkdir()
    (tmp_path / "float").mkdir()
    write_records(tmp_path / "log" / "gridV.nc", m, "depthv", nrec,
                  {"vomecrty": (vs, {"scale_factor": np.float32(1.0e-4), "missing_value": np.int16(SP), "savelog10": np.int32(1)})})
    vals, info = dump(tmp_path / "log" / "gridV.nc", "vomecrty")
    assert not info["packed"]
    vals = vals.reshape((nrec, m.nz, m.ny, m.nx))
    write_records(tmp_path / "float" / "gridV.nc", m, "depthv", nrec,
                  {"vomecrty": ([vals[r, :-1] for r in range(nrec)], {"missing_value": np.float32(SP)})})
    for sub in ("log", "float"):
        ncfiles.write_mesh(m, tmp_path / sub)
        _run(tools["cdfmoc_gpu"], ["-v", "gridV.nc"], tmp_path / sub)
    assert (tmp_path / "log" / "moc.nc").read_bytes() == (tmp_path / "float" / "moc.nc").read_bytes()
