"""16-bit packed records (NC_SHORT + scale_factor / add_offset, as cdf16bit writes them): the decode the device applies
(K3b, cdftools_b200/csrc/unpack_kernels.cuh) restated in NumPy, and checked bit for bit against the host reader's
nc3::Reader::read_f32 (getvar's three masked passes, src/cdfio.F90:1599-1605) on adversarial inputs.  CPU only."""
import json
import subprocess
from pathlib import Path

import numpy as np
import pytest
from scipy.io import netcdf_file

HERE = Path(__file__).resolve().parent
SRC = HERE / "helpers" / "unpack_dump.cpp"


def unpack_i16(raw, sf, ao, sp):
    """int16 -> float32, then x*sf where x != sp (if sf != 1), then x+ao where x != sp (if ao != 0), all in float32: the
    offset pass compares the SCALED value with the missing value."""
    sf, ao, sp = np.float32(sf), np.float32(ao), np.float32(sp)
    x = np.asarray(raw, np.int16).astype(np.float32)
    if sf != np.float32(1):
        x = np.where(x != sp, x * sf, x).astype(np.float32)
    if ao != np.float32(0):
        x = np.where(x != sp, x + ao, x).astype(np.float32)
    return x


def write_packed(path, raw, sf=None, ao=None, sp=None, sp_name="missing_value", savelog10=False):
    f = netcdf_file(str(path), "w", version=2)
    f.createDimension("x", raw.size)
    v = f.createVariable("v", "h", ("x",))
    v[:] = raw
    if sf is not None:
        v.scale_factor = np.float32(sf)
    if ao is not None:
        v.add_offset = np.float32(ao)
    if sp is not None:
        setattr(v, sp_name, np.int16(sp))
    if savelog10:
        v.savelog10 = np.int32(1)
    f.close()


def build_unpack_dump(outdir):
    """Compiles tests/helpers/unpack_dump.cpp into outdir; returns run(path, var) -> (values as read_f32 gives them, the
    packed_i16 query as a dict)."""
    exe = Path(outdir) / "unpack_dump"
    subprocess.run(["g++", "-O2", "-std=c++17", "-pthread", "-ffp-contract=off", "-o", str(exe), str(SRC)], check=True)

    def run(path, var="v"):
        out = Path(str(path) + ".bin")
        r = subprocess.run([str(exe), str(path), var, str(out)], capture_output=True, text=True, check=True)
        return np.fromfile(out, np.float32), json.loads(r.stdout)
    return run


@pytest.fixture(scope="module")
def dump(tmp_path_factory):
    return build_unpack_dump(tmp_path_factory.mktemp("unpack_dump"))


_RNG = np.random.default_rng(20261020)
_EXTREMES = np.array([-32768, 32767, -32767, 0, 1, -1], np.int16)
CASES = {
    # values equal to the missing value stay as they are
    "missing": (np.array([5, -32767, 7, -32767, 0, 32767, -32768], np.int16), 0.001, 20.0, -32767),
    # 200 * 0.5 == 100 == spval: the scaled value equals the missing value, so the offset is skipped
    "scaled_hits_missing": (np.array([200, 100, 201, -200, 199], np.int16), 0.5, 3.25, 100),
    "sf_one_ao_set": (np.array([0, 1, 2, 9999, -4, 32767], np.int16), 1.0, 273.15, 9999),
    "sf_set_ao_zero": (np.array([0, 1, 2, 9999, -4, -32768], np.int16), 0.0015259022, 0.0, 9999),
    "extremes": (_EXTREMES, 0.0001, -1.5, 0),
    "odd_1": (np.array([12345], np.int16), 0.002, 15.0, -32768),
    "odd_9": (_RNG.integers(-32768, 32768, 9).astype(np.int16), 0.00045, 35.0, -32768),
    "odd_1001": (_RNG.integers(-32768, 32768, 1001).astype(np.int16), 1.1e-4, -2.7, 0),
    "tiny_sf": (_RNG.integers(-32768, 32768, 333).astype(np.int16), 1.0e-40, 0.0, 7),   # subnormal products
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_restatement_equals_host_reader_bitwise(dump, tmp_path, case):
    raw, sf, ao, sp = CASES[case]
    raw = np.concatenate([raw, _EXTREMES, np.array([sp], np.int16)])
    p = tmp_path / "p.nc"
    write_packed(p, raw, sf, ao, sp)
    host, info = dump(p)
    assert info["packed"] and np.float32(info["sf"]) == np.float32(sf) and np.float32(info["ao"]) == np.float32(ao)
    assert info["sp"] == float(sp)
    mine = unpack_i16(raw, info["sf"], info["ao"], info["sp"])
    assert host.view(np.uint32).tolist() == mine.view(np.uint32).tolist()


def test_missing_attributes_mean_plain_conversion(dump, tmp_path):
    raw = np.array([-32768, -1, 0, 1, 32767], np.int16)
    p = tmp_path / "p.nc"
    write_packed(p, raw)
    host, info = dump(p)
    assert info == {"packed": True, "sf": 1.0, "ao": 0.0, "sp": 0.0}
    assert np.array_equal(host, raw.astype(np.float32))


def test_fill_value_spelling_is_found(dump, tmp_path):
    raw = np.array([3, -9, 3, 4], np.int16)
    p = tmp_path / "p.nc"
    write_packed(p, raw, 0.25, 1.0, 3, sp_name="_FillValue")
    host, info = dump(p)
    assert info["sp"] == 3.0
    assert np.array_equal(host.view(np.uint32), unpack_i16(raw, 0.25, 1.0, 3).view(np.uint32))


def test_savelog10_is_not_offered_to_the_device(dump, tmp_path):
    p = tmp_path / "p.nc"
    write_packed(p, np.array([1, 2, 3], np.int16), 0.5, 0.0, 0, savelog10=True)
    _, info = dump(p)
    assert info["packed"] is False
