"""cdfmaxmoc's window search (src/cdfmaxmoc.f90:158-167): the C oracle against the NumPy twin, and the rule for
non-finite windows that both follow (gfortran's MAXVAL / MAXLOC, MINVAL / MINLOC):
  * NaN cells are skipped;
  * a window without a non-NaN cell gives NaN, located at its first cell;
  * otherwise the location is the first cell, in (jj fastest, jk) order, holding the extremum -- an all -Inf window
    (max) or all +Inf window (min) included.
The ISO Fortran standard leaves MAXLOC of an all-NaN array processor dependent; the rule above is gfortran's."""
import os
from pathlib import Path

import numpy as np
import pytest

from oracle import np_oracle as npo

NZ, NY = 9, 13
REF = Path(os.environ["CDFTOOLS_REF"]) if os.environ.get("CDFTOOLS_REF") else None


def field(seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((NZ, NY)) * 10).astype(np.float32)


def same(a, b):
    """Two results equal: values bit for bit (any NaN equals any NaN), locations exactly."""
    for x, y in zip(a[:2], b[:2]):
        x, y = np.float32(x), np.float32(y)
        if not ((np.isnan(x) and np.isnan(y)) or x.view(np.int32) == y.view(np.int32)):
            return False
    return tuple(a[2]) == tuple(b[2]) and tuple(a[3]) == tuple(b[3])


def check(oracle_mod, r, win):
    got, ref = oracle_mod.maxmoc(r, *win), npo.maxmoc(r, *win)
    assert same(got, ref), (win, got, ref)
    return got


def cases():
    """(name, rmoc (nz, ny), window (ijmin, ijmax, ikmin, ikmax)) -- 1-based inclusive windows."""
    full = (1, NY, 1, NZ)
    out = []
    r = field(1)
    out += [("random-full", r, full), ("random-sub", r, (3, 11, 2, 7)), ("one-cell", r, (5, 5, 4, 4)),
            ("one-row", r, (1, NY, 6, 6)), ("one-column", r, (7, 7, 1, NZ))]
    r = np.round(field(2) / 8).astype(np.float32)          # small integers: many exact ties
    out += [("ties", r, full)]
    r = np.zeros((NZ, NY), np.float32)
    r[::2, 1::3] = -0.0                                     # a +0 / -0 plateau, as over land
    out += [("zero-plateau", r, full), ("zero-plateau-sub", r, (2, 9, 3, 8))]
    r = np.where(field(3) > 0, np.float32(-0.0), np.float32(0.0)).astype(np.float32)
    r[4, 6] = -1.0
    out += [("signed-zeros", r, full)]
    r = field(4)
    r[[0, 3, 8], [2, 7, 12]] = np.nan
    out += [("few-nan", r, full)]
    r = field(5)
    r[0, 0] = r[NZ - 1, NY - 1] = np.nan
    out += [("nan-first-and-last", r, full), ("nan-first-cell", r, (1, 4, 1, 3)), ("nan-last-cell", r, (10, NY, 7, NZ))]
    r = np.full((NZ, NY), np.nan, np.float32)
    out += [("all-nan", r, full), ("all-nan-sub", r, (4, 6, 2, 2))]
    r = field(6)
    r[:, 5] = np.nan                                        # one latitude poisoned at every level
    out += [("all-nan-latitude", r, (6, 6, 1, NZ))]
    out += [("all-minus-inf", np.full((NZ, NY), -np.inf, np.float32), (2, 7, 3, 5)),
            ("all-plus-inf", np.full((NZ, NY), np.inf, np.float32), (2, 7, 3, 5))]
    r = np.full((NZ, NY), -np.inf, np.float32)
    r[2, 3:6] = np.nan
    out += [("minus-inf-and-nan", r, full)]
    r = field(7)
    r[1, 2], r[4, 4], r[6, 9], r[7, 1] = np.inf, -np.inf, np.nan, np.inf
    out += [("mixed-inf-nan", r, full)]
    r = np.full((NZ, NY), np.nan, np.float32)
    r[5, 8] = np.inf
    r[6, 2] = -np.inf
    out += [("inf-among-nan", r, full)]
    return out


CASES = cases()


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_maxmoc_c_equals_numpy(oracle_mod, case):
    _, r, win = case
    check(oracle_mod, r, win)


def test_maxmoc_rule_on_non_finite_windows(oracle_mod):
    """What the rule gives, spelled out case by case."""
    nan = np.full((NZ, NY), np.nan, np.float32)
    vmax, vmin, lmax, lmin = check(oracle_mod, nan, (4, 6, 2, 3))
    assert np.isnan(vmax) and np.isnan(vmin) and lmax == (4, 2) and lmin == (4, 2)
    ninf = np.full((NZ, NY), -np.inf, np.float32)
    vmax, vmin, lmax, lmin = check(oracle_mod, ninf, (2, 7, 3, 5))
    assert vmax == -np.inf and vmin == -np.inf and lmax == (2, 3) and lmin == (2, 3)
    ninf[3, 1] = np.nan                                     # NaN at the first cell is skipped
    ninf[3, 2] = np.nan
    vmax, _, lmax, lmin = check(oracle_mod, ninf, (2, 7, 4, 5))
    assert vmax == -np.inf and lmax == (4, 4) and lmin == (4, 4)
    r = field(8)
    r[0, 0], r[0, 1] = np.nan, np.float32(1e30)
    r[NZ - 1, NY - 1] = np.float32(-1e30)
    vmax, vmin, lmax, lmin = check(oracle_mod, r, (1, NY, 1, NZ))
    assert vmax == np.float32(1e30) and lmax == (2, 1) and vmin == np.float32(-1e30) and lmin == (NY, NZ)
    r = np.zeros((NZ, NY), np.float32)
    r[0, 0] = -0.0
    vmax, vmin, lmax, lmin = check(oracle_mod, r, (1, NY, 1, NZ))
    assert lmax == (1, 1) and lmin == (1, 1) and np.signbit(vmax) and np.signbit(vmin)


def test_maxmoc_finite_windows_unchanged(oracle_mod):
    """Finite data: the first strictly greater / smaller value wins, as a plain sequential scan finds it."""
    for seed in range(20):
        r = np.round(field(100 + seed) / 4).astype(np.float32)
        rng = np.random.default_rng(seed)
        j0, k0 = int(rng.integers(1, NY + 1)), int(rng.integers(1, NZ + 1))
        win = (j0, int(rng.integers(j0, NY + 1)), k0, int(rng.integers(k0, NZ + 1)))
        vmax, vmin, lmax, lmin = check(oracle_mod, r, win)
        w = r[win[2] - 1:win[3], win[0] - 1:win[1]]
        assert vmax == w.max() and vmin == w.min()
        kk, jj = np.unravel_index(np.argmax(w), w.shape)     # argmax / argmin: first occurrence in C order
        assert lmax == (win[0] + jj, win[2] + kk)
        kk, jj = np.unravel_index(np.argmin(w), w.shape)
        assert lmin == (win[0] + jj, win[2] + kk)


@pytest.mark.skipif(REF is None or not (REF / "src" / "cdfmaxmoc.f90").exists(),
                    reason="needs the CDFTOOLS sources ($CDFTOOLS_REF)")
def test_reference_uses_the_intrinsics():
    """The rule above is that of the Fortran intrinsics: cdfmaxmoc must call them, not a hand-written loop."""
    src = (REF / "src" / "cdfmaxmoc.f90").read_text(errors="replace").upper()
    for name in ("MAXVAL", "MINVAL", "MAXLOC", "MINLOC"):
        assert name + "(" in src.replace(" (", "("), name
