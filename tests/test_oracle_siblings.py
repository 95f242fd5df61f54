"""Sibling tools (SURVEY.md section 8 f3): the C restatements of cdfzonalsum / cdfzonalmean / cdfmhst against independent
NumPy restatements (bit for bit) and against closed-form cases.  CPU only."""
import numpy as np
import pytest

import oracle
from oracle import np_oracle as npo


def _case(seed, nx=41, ny=9, nk=5):
    rng = np.random.default_rng(seed)
    e1 = (rng.random((ny, nx)) * 1e4 + 1e3).astype(np.float32)
    e2 = (rng.random((ny, nx)) * 1e4 + 1e3).astype(np.float32)
    msk = (rng.random((nk, ny, nx)) > 0.3).astype(np.float32)
    atl = (rng.random((ny, nx)) > 0.6).astype(np.float32)
    ind = (rng.random((ny, nx)) > 0.7).astype(np.float32)
    pac = (rng.random((ny, nx)) > 0.5).astype(np.float32)
    zv = rng.standard_normal((nk, ny, nx)).astype(np.float32)
    return e1, e2, msk, atl, ind, pac, zv, rng


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("basins", [True, False])
def test_zonalsum_c_equals_numpy(seed, basins):
    e1, e2, msk, atl, ind, pac, zv, rng = _case(seed)
    zm = oracle.zonal_masks(msk[0], atl, ind, pac) if basins else oracle.zonal_masks(msk[0])
    assert zm.shape[2] == (5 if basins else 1)
    if basins:   # indo-pacific = ind + pac clipped to 1 (cdfzonalsum.f90:292-295)
        assert np.array_equal(zm[:, :, 2], np.minimum(atl * 0 + ind + pac, 1).astype(np.float32))
    alpha = (rng.random(e1.shape[0]) + 0.5).astype(np.float32)
    a = oracle.zonalsum_record(zm, msk, zv, oracle.zonal_dlsurf(e1, e2), alpha)
    b = npo.zonalsum_record(zm, msk, zv, e1, e2, alpha)
    assert np.array_equal(a, b)


@pytest.mark.parametrize("seed", [0, 3])
@pytest.mark.parametrize("lmax", [False, True])
def test_zonalmean_c_equals_numpy(seed, lmax):
    e1, e2, msk, atl, ind, pac, zv, rng = _case(seed)
    msk[:, 2, :] = 0   # a fully masked row: mean, max, min = zspval (cdfzonalmean.f90:331-342)
    zm = oracle.zonal_masks(msk[0], atl, ind, pac)
    a = oracle.zonalmean_record(zm, msk, zv, oracle.zonal_dlsurf(e1, e2), -9.5, lmax)
    b = npo.zonalmean_record(zm, msk, zv, e1, e2, -9.5, lmax)
    assert np.array_equal(a[0], b[0])
    assert np.all(a[0][:, :, 2] == -9.5)
    if lmax:
        assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
        assert np.all(a[1][:, :, 2] == np.float32(-9.5)) and np.all(a[2][:, :, 2] == np.float32(-9.5))
    else:
        assert a[1] is None and a[2] is None


def _nan_rows():
    """Rows of one level (nx = 8, every mask 1 unless stated) with NaN cells in every position that matters to the
    zonal max / min -> (zv, zmaskvar) of shape (1, ny, 8)."""
    nan = np.nan
    rows = [[5, 1, 2, nan, 3, -1, 0.5, 0.25],        # NaN after the max, before the min
            [1, 2, nan, 9, 3, -4, 0.5, 2],           # NaN before the max
            [nan, 1, 2, 3, -2, 4, 0.5, 1],           # i = 0
            [1, 2, 3, -2, 4, 0.5, 1, nan],           # i = nx-1
            [nan] * 8,                               # every cell
            [0, nan, 0, 2, nan, 0, -3, 0],           # with exact zeros (left out of the minimum)
            [nan, 0, nan, 0, nan, 0, nan, 0],        # NaN and zeros only: max 0, no minimum
            [nan, 1, 2, nan, 3, 4, nan, 5],          # the NaN cells are the wet ones (zmaskvar below)
            [-1, -2, nan, -3, -0.5, nan, -4, -1]]    # all negative: the max comes from a number, not -1.e20
    zv = np.array(rows, np.float32)[None]
    mv = np.ones_like(zv)
    mv[0, 7] = [1, 0, 0, 1, 0, 0, 1, 0]
    return zv, mv


def test_zonalmean_nan_never_changes_max_min(oracle_mod):
    """A NaN cell never changes the zonal max / min (include/cdfgpu.h), in the C oracle and the NumPy twin alike; the
    mean of a row with a NaN stays NaN.  Finite cells keep the bits they had without the rule."""
    zv, mv = _nan_rows()
    ny, nx = zv.shape[1:]
    e1, e2 = np.ones((ny, nx), np.float32), np.full((ny, nx), 2.0, np.float32)
    zm = np.ones((ny, nx, 1), np.float32)
    a = oracle_mod.zonalmean_record(zm, mv, zv, oracle_mod.zonal_dlsurf(e1, e2), -9.5, True)
    b = npo.zonalmean_record(zm, mv, zv, e1, e2, -9.5, True)
    for x, y in zip(a, b):
        assert np.array_equal(x, y, equal_nan=True) and np.array_equal(np.signbit(x), np.signbit(y))
    mean, zmax, zmin = (x[0, 0] for x in a)
    assert np.all(np.isnan(mean))
    big = 1.e20
    assert np.array_equal(zmax, np.array([5, 9, 4, 4, -big, 2, 0, 0, -0.5], np.float32))   # by hand
    assert np.array_equal(zmin, np.array([-1, -4, -2, -2, big, -3, big, big, -4], np.float32))


def test_zonalmean_nan_rule_issue_example(oracle_mod):
    """The row of the rule's statement: zv = [5, 1, 2, NaN, 3, -1, 0.5, 0.25] -> mean NaN, max 5.0, min -1.0."""
    zv = np.array([[[5, 1, 2, np.nan, 3, -1, 0.5, 0.25]]], np.float32)
    one = np.ones((1, 8), np.float32)
    zm, mv = np.ones((1, 8, 1), np.float32), np.ones_like(zv)
    for mean, zmax, zmin in (oracle_mod.zonalmean_record(zm, mv, zv, oracle_mod.zonal_dlsurf(one, one), 0.0, True),
                             npo.zonalmean_record(zm, mv, zv, one, one, 0.0, True)):
        assert np.isnan(mean[0, 0, 0]) and zmax[0, 0, 0] == 5.0 and zmin[0, 0, 0] == -1.0


def test_zonalmean_of_a_constant_is_the_constant():
    e1, e2, msk, atl, ind, pac, zv, rng = _case(5)
    zm = oracle.zonal_masks(np.ones_like(msk[0]))
    mean, zmax, zmin = oracle.zonalmean_record(zm, np.ones_like(msk), np.full_like(zv, 2.5), oracle.zonal_dlsurf(e1, e2), 0.0, True)
    assert np.allclose(mean, 2.5, rtol=1e-14)
    assert np.all(zmax == 2.5) and np.all(zmin == 2.5)


@pytest.mark.parametrize("zdim", [False, True])
@pytest.mark.parametrize("basins", [True, False])
def test_mhst_c_equals_numpy(zdim, basins):
    e1, e2, msk, atl, ind, pac, zvt, rng = _case(7)
    e3 = (rng.random(zvt.shape) * 100 + 1).astype(np.float32)
    zvs = rng.standard_normal(zvt.shape).astype(np.float32)
    kw = dict(atl=atl, pac=pac, ind=ind) if basins else {}
    h1, s1 = oracle.mhst_record(e1, e3, msk[0], zvt, zvs, zdim=zdim, **kw)
    h2, s2 = npo.mhst_record(e1, e3, msk[0], zvt, zvs, zdim=zdim, **kw)
    assert np.array_equal(h1, h2) and np.array_equal(s1, s2)
    if not basins:
        assert np.all(h1[:, 1:] == 0)
    if zdim:   # the last level of the cumulative output is the non-zdim result
        h3, s3 = oracle.mhst_record(e1, e3, msk[0], zvt, zvs, zdim=False, **kw)
        assert np.array_equal(h1[-1], h3[0]) and np.array_equal(s1[-1], s3[0])


def test_mhst_global_sum_skips_first_and_last_column():
    e1, e2, msk, atl, ind, pac, zvt, rng = _case(9)
    e3 = np.ones_like(zvt)
    ones = np.ones_like(msk[0])
    zvs = np.zeros_like(zvt)
    zvs[:, :, 0] = 7.0
    zvs[:, :, -1] = 7.0
    h, s = oracle.mhst_record(np.ones_like(e1), e3, ones, zvs, zvs, atl=ones, pac=ones, ind=ones)
    assert np.all(s[0, 0] == 0)                      # global: i = 2..npiglo-1 only (cdfmhst.f90:343)
    assert np.all(s[0, 1] == 2 * 7.0 * zvt.shape[0])  # basins: all i
