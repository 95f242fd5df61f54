"""Pins the oracle's EOS on the only known-answer values the reference holds (comments in src/eos.f90)."""
import numpy as np
import pytest

from oracle import np_oracle as npo


def test_kat_eos80_insitu(oracle_mod):
    # src/eos.f90:820  rho = 1028.35011066567 kg/m^3 for z=3000 dbar, pt=3 Celsius, sp=35.5 psu (value of dlr, :879)
    assert abs(oracle_mod.eos_dlr(3.0, 35.5, 3000.0, False) - 1028.35011066567) < 5e-12 * 1028
    assert abs(float(npo.eos_dlr(np.float32(3.0), np.float32(35.5), 3000.0, False)) - 1028.35011066567) < 5e-12 * 1028


def test_kat_teos10_insitu(oracle_mod):
    # src/eos.f90:817  rho = 1028.21993233072 kg/m^3 for z=3000 dbar, ct=3 Celsius, sa=35.5 g/kg
    assert abs(oracle_mod.eos_dlr(3.0, 35.5, 3000.0, True) - 1028.21993233072) < 5e-12 * 1028
    assert abs(float(npo.eos_dlr(np.float32(3.0), np.float32(35.5), 3000.0, True)) - 1028.21993233072) < 5e-12 * 1028


def test_kat_neutral(oracle_mod):
    # src/eos.f90:646  rho(20,35) = 1024.59416751197 kg/m^3 (-1000 in the returned value)
    v = oracle_mod.sigmantr(np.array([20.0], np.float32), np.array([35.0], np.float32))[0]
    assert abs(v - 24.59416751197) < 5e-11
    assert npo.sigmantr(np.array([20.0], np.float32), np.array([35.0], np.float32))[0] == v


def test_derived_kats(oracle_mod):
    # SURVEY.md section 4: values re-derived from the formulas at survey time
    f = lambda t, s, p, teos=False: oracle_mod.sigmai_dep(np.array([t], np.float32), np.array([s], np.float32), p, teos)[0]
    assert f(3.0, 35.5, 3000.0) == 41.83636437682958
    assert f(3.0, 35.5, 3000.0, True) == 41.706186041879164
    assert f(20.0, 35.0, 0.0) == 24.765493039434205
    assert f(10.0, 35.0, 0.0) == 26.95427774818063
    assert f(2.0, 34.9, 2000.0) == 37.092842616970984


def test_land_is_zero(oracle_mod):
    # dltm = 0 where S == 0 (src/eos.f90:852-856)
    out = oracle_mod.sigmai_dep(np.array([0.0, 5.0], np.float32), np.array([0.0, 0.0], np.float32), 2000.0)
    assert np.all(out == 0.0)


def test_c_vs_numpy_bit_exact(oracle_mod):
    rng = np.random.default_rng(1)
    t = rng.uniform(-2.5, 33.0, 200_000).astype(np.float32)
    s = rng.uniform(0.0, 42.0, 200_000).astype(np.float32)
    s[::11] = 0.0
    for pref in (0.0, 1000.0, 2000.0, 4321.0):
        for teos in (False, True):
            assert np.array_equal(oracle_mod.sigmai_dep(t, s, pref, teos), npo.sigmai_dep(t, s, pref, teos))
    assert np.array_equal(oracle_mod.sigmantr(t, s), npo.sigmantr(t, s))


def test_sigma0_equals_pref0_and_dlr0_only(oracle_mod):
    # sigma0 == sigmai(pref=0) (src/eos.f90:630) -- and with dlh == 0 only dlr0 survives, exactly
    rng = np.random.default_rng(2)
    t = rng.uniform(-2, 30, 1000).astype(np.float32)
    s = rng.uniform(30, 40, 1000).astype(np.float32)
    full = oracle_mod.sigmai_dep(t, s, 0.0)
    E = npo._COEF["EOS80"]
    tt = t.astype(np.float64) * (1.0 / 40.0)
    ss = np.sqrt(np.abs(s.astype(np.float64) + 20.0) * (1.0 / 40.0))
    assert np.array_equal(full, (npo._poly_k(E, 0, tt, ss) + 0.0) - 1000.0)


def test_coefficient_header_matches_the_reference_source(tmp_path):
    """include/cdf_eos_coeffs.h is DATA extracted from the reference (tools/gen_eos_coeffs.py, src/eos.f90:214-279,
    408-466).  Where the CDFTOOLS sources are at hand ($CDFTOOLS_REF) the header is regenerated and compared; skipped
    without them."""
    import os
    import subprocess
    import sys
    from pathlib import Path
    if not os.environ.get("CDFTOOLS_REF") or not (Path(os.environ["CDFTOOLS_REF"]) / "src" / "eos.f90").exists():
        pytest.skip("needs the CDFTOOLS sources ($CDFTOOLS_REF)")
    root = Path(__file__).resolve().parent.parent
    out = tmp_path / "cdf_eos_coeffs.h"
    subprocess.run([sys.executable, str(root / "tools" / "gen_eos_coeffs.py"), str(out)], check=True, capture_output=True)
    assert out.read_text() == (root / "include" / "cdf_eos_coeffs.h").read_text()
