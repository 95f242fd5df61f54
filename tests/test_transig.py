"""cdftransig_xy3d (SURVEY.md section 8 f3): C oracle = NumPy twin bit for bit, the host-side bin table of the product
against both, and -- on the B200 box -- kernel K6 through the C ABI against the oracle (every transport lands in the
reference's class and the accumulators are bit for bit the oracle's)."""
import numpy as np
import pytest

from cdftools_b200 import lib as cdflib
from cdftools_b200 import synth
from oracle import np_oracle as npo

CODES = [(101, 23.0, 0.03, 999.0, 999.0), (93, 24.2, 0.10, 32.3, 0.05), (88, 24.5, 0.10, 999.0, 999.0),
         (174, 29.0, 0.05, 999.0, 999.0), (20, 25.0, 0.2, 27.5, 0.07)]


@pytest.mark.parametrize("code", CODES)
def test_bin_table_three_ways(oracle_mod, code):
    a, b, c = oracle_mod.transig_bins(*code), npo.transig_bins(*code), cdflib.transig_bins(*code)
    for x, y, z in zip(a[:3], b[:3], c[:3]):
        assert np.array_equal(x, y) and np.array_equal(x, z)
    assert a[3] == b[3] == c[3]
    assert a[2].min() >= 1 and a[2].max() == code[0]          # the presets leave no hole in the table
    assert np.all(np.diff(a[2]) >= 0)


def test_code_presets_match_reference_table():
    # src/cdftransig_xy3d.f90:188-197
    assert cdflib.TRANSIG_CODES["1000"] == (1000.0, 93, 24.2, 0.10, 32.3, 0.05)
    assert cdflib.TRANSIG_CODES["0"][1:4] == (101, 23.0, 0.03) and cdflib.TRANSIG_CODES["2000"][1] == 174


def frames(m, n):
    out = []
    for r in range(n):
        zu = synth.make_v_record(m, 10 + r)[:-1] * m.umask[:-1]
        zv = synth.make_v_record(m, r)[:-1] * m.vmask[:-1]
        zt, zs = (x[:-1] for x in synth.make_ts_record(m, r))
        out.append((zu.astype(np.float32), zv.astype(np.float32), zt, zs))
    return out


def run_oracle(f, m, fr, pref, code, lperio, teos10=False, first_tag=2):
    nb, smin = code[0], code[1]
    _, _, itab, scm = npo.transig_bins(*code)
    du, dv = np.zeros((nb, m.ny, m.nx)), np.zeros((nb, m.ny, m.nx))
    mu, mv = np.zeros(fr[0][0].shape, np.uint8), np.zeros(fr[0][0].shape, np.uint8)
    e2u = (m.e1u * np.float32(0.9)).astype(np.float32)
    for n, (zu, zv, zt, zs) in enumerate(fr):
        f(e2u, m.e1v, m.e3v_0[:-1], m.e3v_0[:-1] * np.float32(1.01), zu, zv, zt, zs, pref, smin, scm, itab, nb, du, dv, mu, mv,
          n < first_tag, lperio, teos10)
    return du, dv


@pytest.mark.parametrize("grid", ["TINY", "ODD", "SMALL"])
@pytest.mark.parametrize("cfg", [(0.0, CODES[0], False), (1000.0, CODES[1], True), (2000.0, CODES[3], True)])
def test_c_vs_numpy_bit_exact(oracle_mod, grid, cfg):
    pref, code, lperio = cfg
    m = synth.make_mesh(grid)
    fr = frames(m, 3)
    a = run_oracle(oracle_mod.transig_record, m, fr, pref, code, lperio)
    b = run_oracle(npo.transig_record, m, fr, pref, code, lperio)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert np.count_nonzero(a[0]) > 0 and np.count_nonzero(a[1]) > 0


def test_total_transport_is_conserved(oracle_mod):
    # summing over the classes gives back the depth-integrated transport of every column (fp64 rounding only)
    m = synth.make_mesh("SMALL")
    fr = frames(m, 1)
    du, dv = run_oracle(oracle_mod.transig_record, m, fr, 1000.0, CODES[1], False)
    zu, zv = fr[0][0], fr[0][1]
    e2u = (m.e1u * np.float32(0.9)).astype(np.float32)
    tot = (e2u[None] * (zu * m.e3v_0[:-1])).astype(np.float64).sum(axis=0)
    assert np.allclose(du.sum(axis=0), tot, rtol=1e-12, atol=1e-6)


# ---------------------------------------------------------------------------------------------- CUDA path (B200 box)
@pytest.mark.gpu
@pytest.mark.parametrize("grid", ["TINY", "ODD", "SMALL", "ORCA2"])
@pytest.mark.parametrize("cfg", [(0.0, CODES[0], False, False), (1000.0, CODES[1], True, False), (2000.0, CODES[3], True, True),
                                 (1000.0, CODES[4], False, False)])
def test_gpu_parity(gpu_lib, oracle_mod, grid, cfg):
    pref, code, lperio, teos10 = cfg
    m = synth.make_mesh(grid)
    fr = frames(m, 3)
    ref_u, ref_v = run_oracle(oracle_mod.transig_record, m, fr, pref, code, lperio, teos10)
    nb, smin = code[0], code[1]
    _, _, itab, scm = gpu_lib.transig_bins(*code)
    e2u = (m.e1u * np.float32(0.9)).astype(np.float32)
    shape = gpu_lib.cdftransig_setup(e2u, m.e1v, m.e3v_0[:-1], m.e3v_0[:-1] * np.float32(1.01), m.nz, nb, pref, smin, scm, itab,
                                     lperio, teos10)
    for n, (zu, zv, zt, zs) in enumerate(fr):
        gpu_lib.cdftransig_record(zu, zv, zt, zs, set_masks=n < 2)
    du, dv = gpu_lib.cdftransig_fetch(shape)
    # class assignment bit-exact: the sets of (class, j, i) that received transport are identical
    assert np.array_equal(du != 0, ref_u != 0) and np.array_equal(dv != 0, ref_v != 0)
    # each column's accumulators take the frames in order and, within a frame, the levels in order, as the oracle adds
    # them: bit for bit
    assert np.array_equal(du.view(np.int64), ref_u.view(np.int64)) and np.array_equal(dv.view(np.int64), ref_v.view(np.int64))
    gpu_lib.cdftransig_teardown()


@pytest.mark.gpu
def test_gpu_vvl_and_errors(gpu_lib, oracle_mod):
    m = synth.make_mesh("SMALL")
    fr = frames(m, 2)
    code = CODES[1]
    _, _, itab, scm = gpu_lib.transig_bins(*code)
    e2u = (m.e1u * np.float32(0.9)).astype(np.float32)
    e3u, e3v = m.e3v_0[:-1], m.e3v_0[:-1] * np.float32(1.01)
    ref_u, ref_v = run_oracle(oracle_mod.transig_record, m, fr, 1000.0, code, False)
    shape = gpu_lib.cdftransig_setup(e2u, m.e1v, None, None, m.nz, code[0], 1000.0, code[1], scm, itab)
    with pytest.raises(gpu_lib.CdfGpuError):
        gpu_lib.cdftransig_record(*fr[0], set_masks=True)          # -vvl setup: every record must bring e3u / e3v
    for zu, zv, zt, zs in fr:
        gpu_lib.cdftransig_record(zu, zv, zt, zs, True, e3u, e3v)
    du, dv = gpu_lib.cdftransig_fetch(shape)
    assert np.allclose(du, ref_u, rtol=1e-12, atol=1e-9) and np.allclose(dv, ref_v, rtol=1e-12, atol=1e-9)
    bad = itab.copy()
    bad[0] = code[0] + 1
    with pytest.raises(gpu_lib.CdfGpuError):
        gpu_lib.cdftransig_setup(e2u, m.e1v, e3u, e3v, m.nz, code[0], 1000.0, code[1], scm, bad)
