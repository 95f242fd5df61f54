"""The options layered on K1 and K2 against the C oracle at production widths and at the shapes and values where they
could go wrong: cdfmoc -decomp (csrc/moc_decomp.cuh + K1 noscan), cdfmocsig -isodep (K2's ISO instantiation) and the
cdfmaxmoc window search (moc_window_extrema_kernel).

-decomp and -isodep sum in a different order from the reference (warp trees, histograms per warp), so the streamfunctions
are compared with util.assert_psi_close (NaN and Inf patterns exactly).  The maxmoc search reads REAL(4) values: values
and locations equal the oracle's on the slab the GPU computed, exactly.  Every record is seeded."""
import types

import numpy as np
import pytest

import oracle
from cdftools_b200 import lib, synth
from util import assert_psi_close, case_inputs

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_STATE = 2, 3          # CDFGPU_ERR_ARG, CDFGPU_ERR_STATE
F4 = np.float32


@pytest.fixture(scope="module", autouse=True)
def _ctx(gpu_lib, oracle_mod):
    """The session-wide library context (conftest.gpu_lib), never finalised here: the test modules that follow use it."""
    yield


@pytest.fixture(scope="module")
def orca025():
    return synth.make_mesh("ORCA025")


# ---- cdfmoc -decomp -----------------------------------------------------------------------------------------------------
def mesh_case(m, ib=None, teos10=False):
    """A -decomp plan from a synthetic mesh: ib defaults to the 5-basin set, e3m = e3v_0 * vmask."""
    ib5, e3m = case_inputs(oracle, m, synth)
    return types.SimpleNamespace(e1v=m.e1v, e1u=m.e1u, gphiv=m.gphiv, gdept=m.gdept_1d, e3m=e3m,
                                 ib=ib5 if ib is None else np.ascontiguousarray(ib, np.int16),
                                 um=m.umask.astype(np.int16), tm=m.tmask.astype(np.int16), teos10=teos10)


def mesh_record(m, rec, adversarial=False):
    t, s = synth.make_ts_record(m, rec)
    return synth.make_v_record(m, rec, adversarial)[:-1], t[:-1], s[:-1]


def random_case(nx, ny, nz, nb, seed, teos10=False):
    """Every cell carries data, the border rows and columns included: wet cells (e3m > 0) on all four edges, basin masks
    set on all four edges, random umask / tmask.  -> (plan, record)."""
    rng = np.random.default_rng(seed)
    wet = rng.random((nz, ny, nx)) > 0.2
    ib = (rng.random((ny, nx, nb)) > 0.4).astype(np.int16)
    ib[0], ib[-1], ib[:, 0], ib[:, -1] = 1, 1, 1, 1
    lat = np.linspace(-60.0, 70.0, ny) + 0.37
    c = types.SimpleNamespace(
        e1v=(rng.random((ny, nx)) * 4e4 + 5e3).astype(F4), e1u=(rng.random((ny, nx)) * 4e4 + 5e3).astype(F4),
        gphiv=np.ascontiguousarray(np.broadcast_to(lat[:, None], (ny, nx)), F4),
        gdept=np.cumsum(rng.random(nz) * 100 + 10).astype(F4),
        e3m=np.where(wet, rng.random((nz, ny, nx)) * 200 + 5, 0).astype(F4), ib=ib,
        um=(rng.random((nz, ny, nx)) > 0.25).astype(np.int16), tm=wet.astype(np.int16), teos10=teos10)
    rec = ((0.1 * rng.standard_normal((nz - 1, ny, nx))).astype(F4), (rng.random((nz - 1, ny, nx)) * 20 + 2).astype(F4),
           (rng.random((nz - 1, ny, nx)) * 2 + 34).astype(F4))
    return c, rec


def decomp_ref(c, rec, e3m=None):
    with np.errstate(all="ignore"):
        return oracle.cdfmoc_decomp_record(c.e1v, c.e1u, c.gphiv, c.gdept, c.e3m if e3m is None else e3m, c.ib, c.um, c.tm,
                                           *rec, teos10=c.teos10)


def decomp_setup(c):
    shape = lib.cdfmoc_setup(c.e1v, c.e3m, c.ib)
    lib.cdfmoc_decomp_setup(c.e1u, c.gphiv, c.gdept, c.um, c.tm, teos10=c.teos10)
    return shape


def decomp_run(shape, rec, slot=0, jt=0):
    lib.cdfmoc_decomp_submit(slot, jt, *(np.ascontiguousarray(a) for a in rec))
    return lib.cdfmoc_decomp_fetch(slot, shape)


def check_decomp(got, ref, what, rows=None):
    for k in ("total", "bt", "sh", "ag"):
        g = got[k] if rows is None else got[k][:, rows]
        assert_psi_close(g, ref[k], f"{what}: {k}")


def decomp_case(c, rec, what):
    got = decomp_run(decomp_setup(c), rec)
    ref = decomp_ref(c, rec)
    check_decomp(got, ref, what)
    return got, ref


def basins_from_five(ib5, nb):
    """nb = 1..8 basin planes assembled from the 5-basin set (global, atl, inp, ind, pac): binary, distinct."""
    g, atl, inp, ind, pac = (ib5[:, :, b] for b in range(5))
    planes = [g, atl, inp, ind, pac, atl | pac, atl | ind, g & (1 - atl)]
    return np.ascontiguousarray(np.stack(planes[:nb], axis=2), np.int16)


@pytest.mark.parametrize("nb", range(1, 9))
def test_decomp_basin_counts(nb):
    """Every decomp_weighted_t<NB> instantiation; nb = 1 is the run without basins."""
    m = synth.make_mesh("SMALL")
    c = mesh_case(m, basins_from_five(case_inputs(oracle, m, synth)[0], nb))
    got, ref = decomp_case(c, mesh_record(m, 10 + nb), f"nb={nb}")
    assert np.count_nonzero(ref["bt"][:, :, nb - 1]) > 0 and np.count_nonzero(ref["sh"][:, :, nb - 1]) > 0


def test_decomp_nonbinary_masks():
    """Mask values other than 0 / 1 enter the barotropic product fl32(area * mask) and send K1 down its general path."""
    m = synth.make_mesh("SMALL")
    ib = case_inputs(oracle, m, synth)[0].copy()
    ib[:, :, 1] *= 3
    ib[::2, :, 4] *= -2
    decomp_case(mesh_case(m, ib), mesh_record(m, 21), "non-binary masks")


def test_decomp_vvl_between_records():
    """cdfmoc_set_e3v rewrites the e3m every decomp kernel reads: the record after it equals the oracle run with the new
    e3m, which wets dry cells and dries wet ones."""
    m = synth.make_mesh("SMALL")
    c = mesh_case(m)
    rec = mesh_record(m, 22)
    e3b = (c.e3m * F4(1.0625)).astype(F4)
    dry = c.e3m[: m.nz - 1] == 0
    e3b[: m.nz - 1][dry & (np.arange(m.nx)[None, None, :] % 5 == 0)] = F4(40.0)          # wet some dry cells
    e3b[: m.nz - 1][~dry & (np.arange(m.ny)[None, :, None] % 7 == 3)] = F4(0.0)           # dry some wet ones
    shape = decomp_setup(c)
    check_decomp(decomp_run(shape, rec), decomp_ref(c, rec), "before set_e3v")
    lib.cdfmoc_set_e3v(e3b)
    check_decomp(decomp_run(shape, rec, jt=1), decomp_ref(c, rec, e3b), "after set_e3v")


@pytest.mark.parametrize("shape", [(37, 9, 6), (1, 5, 4), (2, 6, 4), (9, 1, 4), (9, 2, 4), (37, 9, 2)],
                         ids=["37x9x6", "nx1", "nx2", "ny1", "ny2", "nz2"])
def test_decomp_wet_borders(shape):
    """Border cells of the geostrophic velocity keep the last V level read (cdfmoc.f90:357) and are summed by K1 and the
    weighted pass like any other: with wet, basin-covered border rows and columns every cell of nx <= 2 or ny <= 2
    is one of them."""
    nx, ny, nz = shape
    c, rec = random_case(nx, ny, nz, 3, nx * 100 + ny * 10 + nz)
    got, ref = decomp_case(c, rec, f"{shape}")
    assert np.count_nonzero(ref["sh"][: nz - 1]) > 0


def test_decomp_nonfinite_inputs():
    """NaN and +-Inf in V, NaN in T (wet) and in S on land (tmask = 0: zsig0 = fl32(NaN * 0) is still NaN)."""
    m = synth.make_mesh("SMALL")
    c = mesh_case(m)
    v, t, s = (a.copy() for a in mesh_record(m, 23))
    wet = np.argwhere(c.e3m[: m.nz - 1] * (c.ib[None, :, :, 0] != 0) > 0)
    land = np.argwhere(c.tm[: m.nz - 1] == 0)
    v[tuple(wet[50])] = np.nan
    v[tuple(wet[400])] = np.inf
    v[tuple(wet[900])] = -np.inf
    t[tuple(wet[1500])] = np.nan
    s[tuple(land[len(land) // 2])] = np.nan
    got, ref = decomp_case(c, (v, t, s), "non-finite")
    for k in ("total", "bt", "sh", "ag"):
        assert np.isnan(ref[k]).any(), k
        assert np.isfinite(ref[k]).any(), k


@pytest.mark.parametrize("grid", [(1442, 24, 75), (4322, 8, 75)], ids=["orca025-width", "orca12-width"])
def test_decomp_production_widths(grid):
    m = synth.make_mesh(grid)
    decomp_case(mesh_case(m, teos10=grid[0] == 4322), mesh_record(m, 24), f"{grid}")


def window_rows(c, rec, j):
    """The plan and record restricted to rows [j-1, j+3): the stencil of row j reads rows j and j + 1 only, so row j (index
    1 of the window) is an exact sub-problem of the whole grid."""
    w = slice(j - 1, j + 3)
    r2 = lambda a: np.ascontiguousarray(a[w])
    r3 = lambda a: np.ascontiguousarray(a[:, w])
    cw = types.SimpleNamespace(e1v=r2(c.e1v), e1u=r2(c.e1u), gphiv=r2(c.gphiv), gdept=c.gdept, e3m=r3(c.e3m), ib=r2(c.ib),
                               um=r3(c.um), tm=r3(c.tm), teos10=c.teos10)
    return cw, tuple(r3(a) for a in rec)


def test_decomp_orca025_sampled_rows(orca025):
    """A whole ORCA025 L75 record on the GPU; the oracle on 4-row windows around sampled rows.  The window argument is
    checked first on SMALL, against the whole-grid oracle, bit for bit."""
    small = synth.make_mesh("SMALL")
    cs, rs = mesh_case(small), mesh_record(small, 25, adversarial=True)
    whole = decomp_ref(cs, rs)
    for j in (1, 2, 17, small.ny - 3):
        part = decomp_ref(*window_rows(cs, rs, j))
        for k in ("total", "bt", "sh", "ag"):
            assert np.array_equal(part[k][:, 1], whole[k][:, j]), (j, k)
    m = orca025
    c, rec = mesh_case(m), mesh_record(m, 25)
    got = decomp_run(decomp_setup(c), rec)
    for j in (1, 2, 300, 511, 900, m.ny - 3):
        ref = decomp_ref(*window_rows(c, rec, j))
        check_decomp(got, {k: v[:, 1:2] for k, v in ref.items()}, f"ORCA025 row {j}", rows=slice(j, j + 1))


def test_decomp_records_in_a_row():
    """Three records on one slot, then three on two slots in turn (one decomposition in flight at a time)."""
    m = synth.make_mesh("ODD")
    c = mesh_case(m)
    recs = [mesh_record(m, 30 + r, adversarial=r == 1) for r in range(3)]
    refs = [decomp_ref(c, r) for r in recs]
    shape = decomp_setup(c)
    for n, rec in enumerate(recs):
        check_decomp(decomp_run(shape, rec, 0, n), refs[n], f"slot 0 rec {n}")
    for n, rec in enumerate(recs):
        check_decomp(decomp_run(shape, rec, n % 2, 3 + n), refs[n], f"slot {n % 2} rec {n}")


# ---- cdfmocsig -isodep --------------------------------------------------------------------------------------------------
def iso_run(e1v, e3v, ib, gdept, nz, recs, cfg, spv=0.0, spt=0.0, sps=0.0, vvl=False):
    """recs: [(v, t, s, eiv or None, e3v of the record or None)] -> [(moc, depi)] of consecutive submits on slot n % 2."""
    pref, eos, smin, sstp, nbins = cfg
    shape = lib.cdfmocsig_setup(e1v, None if vvl else e3v, ib, nz, nbins, smin, sstp, pref, eos, spv, spt, sps)
    lib.cdfmocsig_set_isodep(gdept)
    outs = []
    for n, (v, t, s, eiv, e3r) in enumerate(recs):
        moc, iso = np.empty(shape), np.empty(shape)
        lib.cdfmocsig_submit(n % 2, n, v, t, s, eiv, e3r)
        lib.cdfmocsig_fetch(n % 2, moc)
        lib.cdfmocsig_fetch_isodep(n % 2, iso)
        outs.append((moc, iso))
    return outs


def iso_ref(e1v, e3v, ib, gdept, v, t, s, cfg, spv=0.0, spt=0.0, sps=0.0, eiv=None):
    pref, eos, smin, sstp, nbins = cfg
    with np.errstate(all="ignore"):
        moc, depi = oracle.cdfmocsig_record_isodep(e1v, e3v, ib, gdept, v, t, s, spv, spt, sps, pref, eos, smin, sstp, nbins)
        if eiv is not None:   # the depths do not depend on V
            moc, _ = oracle.cdfmocsig_record(e1v, e3v, ib, v, t, s, spv, spt, sps, pref, eos, smin, sstp, nbins, zveiv=eiv,
                                             want_bins=False)
    return moc, depi


def check_iso(got, ref, what):
    (moc, iso), (rmoc, riso) = got, ref
    assert_psi_close(moc, rmoc, f"{what}: moc")
    empty = riso == 99999.0
    assert np.array_equal(iso == 99999.0, empty), f"{what}: empty classes differ"
    assert np.array_equal(np.isnan(iso), np.isnan(riso)), f"{what}: NaN depths differ"
    ok = ~empty & ~np.isnan(riso)
    assert np.allclose(iso[ok], riso[ok], rtol=1e-11, atol=1e-9), f"{what}: depths"
    assert ok.any() and empty.any()


def mesh_iso(m, rec, cfg, ib=None, adversarial=False, **kw):
    ib = case_inputs(oracle, m, synth)[0] if ib is None else ib
    v, t, s = mesh_record(m, rec, adversarial)
    got = iso_run(m.e1v, m.e3v_0, ib, m.gdept_1d, m.nz, [(v, t, s, None, None)], cfg, **kw)[0]
    check_iso(got, iso_ref(m.e1v, m.e3v_0, ib, m.gdept_1d, v, t, s, cfg, **kw), f"{m.meta['grid']} {cfg}")
    return got


def bins_for(pref, eos):
    """(sigmin, sigstp, nbins): the reference defaults by pref; for neutral density a range its values fall in."""
    if eos == 2:
        return 25.0, 0.05, 80
    nbins, smin, sstp = oracle.default_bins(pref)
    return smin, sstp, nbins


@pytest.mark.parametrize("pref", [0.0, 2000.0])
@pytest.mark.parametrize("eos", [0, 1, 2], ids=["eos80", "teos10", "neutral"])
@pytest.mark.parametrize("grid", ["ODD", "SMALL"])
def test_isodep_eos_and_pref(grid, eos, pref):
    m = synth.make_mesh(grid)
    mesh_iso(m, 40, (pref, eos, *bins_for(pref, eos)))


def test_isodep_missing_values():
    """Land filled with spv, spt, sps = 1e20, -999, 9999.  The reference sets itmask after the scrub
    (cdfmocsig.f90:383-394), so with sps != 0 every cell has itmask = 1: land inside a basin adds depth weight to the
    class of sigma(0, 0), and the 99999 pattern shows it."""
    m = synth.make_mesh("SMALL")
    ib = case_inputs(oracle, m, synth)[0]
    spv, spt, sps = 1.0e20, -999.0, 9999.0
    v = synth.make_v_record(m, 41, spval=spv)[:-1]
    t, s = synth.make_ts_record(m, 41)
    wet = m.tmask.astype(bool)
    t = np.where(wet, t, F4(spt)).astype(F4)[:-1]
    s = np.where(wet, s, F4(sps)).astype(F4)[:-1]
    cfg = (0.0, 0, 23.0, 0.1, 52)
    kw = dict(spv=spv, spt=spt, sps=sps)
    got = iso_run(m.e1v, m.e3v_0, ib, m.gdept_1d, m.nz, [(v, t, s, None, None)], cfg, **kw)[0]
    ref = iso_ref(m.e1v, m.e3v_0, ib, m.gdept_1d, v, t, s, cfg, **kw)
    check_iso(got, ref, "missing values")
    zero_ref = iso_ref(m.e1v, m.e3v_0, ib, m.gdept_1d, np.where(wet[:-1], v, F4(0)), np.where(wet[:-1], t, F4(0)),
                       np.where(wet[:-1], s, F4(0)), cfg)
    assert not np.array_equal(ref[1] == 99999.0, zero_ref[1] == 99999.0)   # the quirk is visible in the result


def test_isodep_mask_over_land_with_v():
    """A global mask that covers land where V != 0 (adversarial records, no missing values): itmask = 0 there, but the
    transport still counts -- the K2 fast path's drop rule must keep such cells."""
    m = synth.make_mesh("SMALL")
    ib = case_inputs(oracle, m, synth)[0].copy()
    ib[:, :, 0] = 1
    mesh_iso(m, 42, (0.0, 0, 23.0, 0.1, 52), ib=ib, adversarial=True)
    mesh_iso(m, 43, (2000.0, 1, 30.0, 0.05, 158), ib=ib, adversarial=True)


def test_isodep_nonfinite():
    """NaN / +-Inf transports in wet cells send their windows down sig_window_general<., true>: a cell whose transport
    is NaN still adds its depth weight.  NaN in T or S: the reference's bin of a NaN density (clamped to 1)."""
    m = synth.make_mesh("SMALL")
    ib = case_inputs(oracle, m, synth)[0]
    v, t, s = (a.copy() for a in mesh_record(m, 44))
    wet = np.argwhere(m.vmask[: m.nz - 1] * (ib[None, :, :, 0] != 0))     # covered by the global basin, i and j interior
    v[tuple(wet[30])] = np.nan
    v[tuple(wet[300])] = np.inf
    v[tuple(wet[700])] = -np.inf
    t[tuple(wet[1100])] = np.nan
    s[tuple(wet[1500])] = np.nan
    cfg = (0.0, 0, 23.0, 0.1, 52)
    got = iso_run(m.e1v, m.e3v_0, ib, m.gdept_1d, m.nz, [(v, t, s, None, None)], cfg)[0]
    ref = iso_ref(m.e1v, m.e3v_0, ib, m.gdept_1d, v, t, s, cfg)
    assert np.isnan(ref[0]).any()
    check_iso(got, ref, "non-finite")


def test_isodep_eiv_and_vvl():
    m = synth.make_mesh("SMALL")
    ib = case_inputs(oracle, m, synth)[0]
    cfg = (2000.0, 0, 30.0, 0.05, 158)
    v, t, s = mesh_record(m, 45)
    eiv = (0.01 * synth.make_v_record(m, 46)[:-1]).astype(F4)
    got = iso_run(m.e1v, m.e3v_0, ib, m.gdept_1d, m.nz, [(v, t, s, eiv, None)], cfg)[0]
    check_iso(got, iso_ref(m.e1v, m.e3v_0, ib, m.gdept_1d, v, t, s, cfg, eiv=eiv), "-eiv")
    e3a = (m.e3v_0 * F4(1.03125)).astype(F4)
    e3b = (m.e3v_0 * F4(0.96875)).astype(F4)
    got = iso_run(m.e1v, None, ib, m.gdept_1d, m.nz, [(v, t, s, None, np.ascontiguousarray(e3a[:-1])),
                                                      (v, t, s, eiv, np.ascontiguousarray(e3b[:-1]))], cfg, vvl=True)
    check_iso(got[0], iso_ref(m.e1v, e3a, ib, m.gdept_1d, v, t, s, cfg), "-vvl rec 0")
    check_iso(got[1], iso_ref(m.e1v, e3b, ib, m.gdept_1d, v, t, s, cfg, eiv=eiv), "-vvl -eiv rec 1")


def test_isodep_forced_cta_shapes(monkeypatch):
    """CDFGPU_K2_WARPS x CDFGPU_K2_CHUNKS, re-planned by set_isodep: every shape matches the oracle.  With one chunk per
    row the histograms are folded in a fixed order (DESIGN.md section 4 (b)): the same shape twice gives the same bits."""
    m = synth.make_mesh("SMALL")
    ib = case_inputs(oracle, m, synth)[0]
    v, t, s = mesh_record(m, 47)
    cfg = (0.0, 0, 23.0, 0.05, 104)
    ref = iso_ref(m.e1v, m.e3v_0, ib, m.gdept_1d, v, t, s, cfg)
    one_chunk = {}
    for warps in (1, 2, 4, 8, 16):
        for chunks in (1, 3, m.nz - 1):
            monkeypatch.setenv("CDFGPU_K2_WARPS", str(warps))
            monkeypatch.setenv("CDFGPU_K2_CHUNKS", str(chunks))
            got = iso_run(m.e1v, m.e3v_0, ib, m.gdept_1d, m.nz, [(v, t, s, None, None)] * 2, cfg)
            check_iso(got[0], ref, f"warps {warps} chunks {chunks}")
            for a, b in zip(got[0], got[1]):
                assert np.array_equal(a, b), f"warps {warps} chunks {chunks}: not reproducible"
            nkc = -(-(m.nz - 1) // chunks)                     # levels per chunk
            assert lib.cdfmocsig_filter_info()["chunks_per_row"] == -(-(m.nz - 1) // nkc)
            if chunks == 1:
                one_chunk[warps] = got[0]
    differ = [w for w in one_chunk if not all(np.array_equal(a, b) for a, b in zip(one_chunk[w], one_chunk[1]))]
    assert not differ, f"one chunk per row: warps {differ} differ from 1 warp in the last bits"


def distinct_patterns(nx, ny, npat, seed):
    """(ny, nx, 5) masks holding `npat` distinct non-zero tuples (binary up to 31, then non-binary), each on interior cells."""
    rng = np.random.default_rng(seed)
    tuples = [[(p >> b) & 1 for b in range(5)] for p in range(1, 32)] + [[2, 0, 0, 0, p] for p in range(1, 9)]
    ib = np.zeros((ny, nx, 5), np.int16)
    cells = rng.permutation([(j, i) for j in range(1, ny - 1) for i in range(1, nx - 1)])
    for n, (j, i) in enumerate(cells):
        if (7 * j + i) % 11:   # some cells stay outside every basin
            ib[j, i] = tuples[n % npat]
    assert len({tuple(x) for x in ib[:, 1:-1].reshape(-1, 5)}) == npat + 1
    return ib


def smem_bytes(iso, warps, nbins, npat1, nb, tab_rows=8):
    """sig_smem_bytes (api_mocsig.inc): what one CTA of K2 needs."""
    nh = 3 if iso else 1
    doubles = (warps * (nh * nbins * npat1 + tab_rows * 32) + nbins * nb + (nbins + 1) // 2 + 1) & ~1
    return doubles * 8 + 4 * warps * 32 * 16


BUDGET = 227 * 1024 - 2048


def iso_random(nx, ny, nz, ib, seed):
    rng = np.random.default_rng(seed)
    e1v = (rng.random((ny, nx)) * 4e4 + 5e3).astype(F4)
    e3v = (rng.random((nz, ny, nx)) * 200 + 5).astype(F4)
    v = (0.1 * rng.standard_normal((nz - 1, ny, nx))).astype(F4)
    t = (rng.random((nz - 1, ny, nx)) * 26 - 1).astype(F4)
    s = (rng.random((nz - 1, ny, nx)) * 3.5 + 33).astype(F4)
    gdept = np.cumsum(rng.random(nz) * 100 + 10).astype(F4)
    return e1v, e3v, v, t, s, gdept


@pytest.mark.parametrize("npat", [1, 8, 31])
def test_isodep_many_classes_and_patterns(npat):
    """158 sigma2 classes with up to 31 distinct mask tuples (all setup accepts): K2 gives up warps until three histograms
    per warp fit in shared memory (31 tuples: one warp per CTA).  One tuple more is refused by setup."""
    nx, ny, nz = 64, 24, 6
    ib = distinct_patterns(nx, ny, npat, npat)
    e1v, e3v, v, t, s, gdept = iso_random(nx, ny, nz, ib, npat)
    cfg = (2000.0, 0, 30.0, 0.05, 158)
    got = iso_run(e1v, e3v, ib, gdept, nz, [(v, t, s, None, None)], cfg)[0]
    check_iso(got, iso_ref(e1v, e3v, ib, gdept, v, t, s, cfg), f"{npat} patterns")
    if npat == 31:
        assert smem_bytes(True, 1, 158, 31, 5) * 2 > BUDGET          # one warp, one CTA per SM
        with pytest.raises(lib.CdfGpuError) as e:
            lib.cdfmocsig_setup(e1v, e3v, distinct_patterns(nx, ny, 32, 1), nz, 158, 30.0, 0.05, 2000.0, 0)
        assert e.value.code == ERR_ARG


def test_isodep_shared_memory_limit():
    """The largest class count whose three histograms (31 mask tuples) fit in one warp's CTA runs and matches the oracle;
    one class more: set_isodep refuses with CDFGPU_ERR_ARG, leaves -isodep off, and the plain kernel still runs."""
    nx, ny, nz = 64, 24, 6
    ib = distinct_patterns(nx, ny, 31, 5)
    fit = max(n for n in range(100, 1000) if smem_bytes(True, 1, n, 31, 5) <= BUDGET)
    e1v, e3v, v, t, s, gdept = iso_random(nx, ny, nz, ib, 6)
    cfg = (2000.0, 0, 30.0, 0.05, fit)
    got = iso_run(e1v, e3v, ib, gdept, nz, [(v, t, s, None, None)], cfg)[0]
    check_iso(got, iso_ref(e1v, e3v, ib, gdept, v, t, s, cfg), f"{fit} classes")
    over = fit + 1
    shape = lib.cdfmocsig_setup(e1v, e3v, ib, nz, over, 30.0, 0.05, 2000.0, 0)
    with pytest.raises(lib.CdfGpuError) as e:
        lib.cdfmocsig_set_isodep(gdept)
    assert e.value.code == ERR_ARG and "shared memory" in str(e.value)
    moc = np.empty(shape)
    lib.cdfmocsig_submit(0, 0, v, t, s)
    lib.cdfmocsig_fetch(0, moc)
    ref, _ = oracle.cdfmocsig_record(e1v, e3v, ib, v, t, s, 0.0, 0.0, 0.0, 2000.0, 0, 30.0, 0.05, over, want_bins=False)
    assert_psi_close(moc, ref, f"{over} classes without -isodep")
    with pytest.raises(lib.CdfGpuError) as e:
        lib.cdfmocsig_fetch_isodep(0, np.empty(shape))
    assert e.value.code == ERR_STATE


def iso_sampled_rows(m, ib, rec, cfg, rows, whole=None):
    v, t, s = mesh_record(m, rec)
    got = iso_run(m.e1v, m.e3v_0, ib, m.gdept_1d, m.nz, [(v, t, s, None, None)], cfg)[0]
    for j in rows:   # the oracle skips the first and last row it is given: 3-row windows, compare the middle
        w = slice(j - 1, j + 2)
        ref = iso_ref(m.e1v[w], m.e3v_0[:, w], ib[w], m.gdept_1d, v[:, w], t[:, w], s[:, w], cfg)
        moc, iso = got[0][j], got[1][j]
        assert_psi_close(moc, ref[0][1], f"row {j}: moc")
        empty = ref[1][1] == 99999.0
        assert np.array_equal(iso == 99999.0, empty), f"row {j}: empty classes"
        assert np.allclose(iso[~empty], ref[1][1][~empty], rtol=1e-11, atol=1e-9), f"row {j}: depths"
    return got


def test_isodep_orca025_sampled_rows(orca025):
    """ORCA025 L75, sigma0 / 104 classes: 8 warps x 2 CTAs per SM, one chunk per row."""
    m = orca025
    got = iso_sampled_rows(m, case_inputs(oracle, m, synth)[0], 48, (0.0, 0, 23.0, 0.05, 104), (1, 2, 200, 511, 777, 1019))
    assert lib.cdfmocsig_filter_info()["chunks_per_row"] == 1
    assert np.all(got[0][0] == 0.0) and np.all(got[1][0] == 99999.0)


def test_isodep_orca12_band():
    """383 rows of ORCA12 as one domain, sigma2 / 158 classes: a short launch, several chunks per row, fewer warps."""
    m = synth.make_mesh("ORCA12", rows=(1338, 1721))
    iso_sampled_rows(m, case_inputs(oracle, m, synth)[0], 49, (2000.0, 0, 30.0, 0.05, 158), (1, 2, 100, 191, 300, 381))
    assert lib.cdfmocsig_filter_info()["chunks_per_row"] > 1


# ---- cdfmaxmoc ----------------------------------------------------------------------------------------------------------
def same_result(got, ref):
    """Values equal (any NaN equals any NaN; the sign of a zero is not compared), locations exactly."""
    for g, r in zip(got[:2], ref[:2]):
        g, r = F4(g), F4(r)
        if not (g == r or (np.isnan(g) and np.isnan(r))):
            return False
    return tuple(got[2]) == tuple(ref[2]) and tuple(got[3]) == tuple(ref[3])


def check_max(slot, psi, basin, win):
    got = lib.cdfmoc_maxmoc(slot, basin, *win)
    ref = oracle.maxmoc(psi[:, :, basin].astype(F4), *win)
    assert same_result(got, ref), (basin, win, got, ref)
    return got


def moc_slab(e1v, e3m, ib, v, slot=0):
    shape = lib.cdfmoc_setup(e1v, e3m, ib)
    out = np.empty(shape)
    lib.cdfmoc_submit(slot, 0, np.ascontiguousarray(v))
    lib.cdfmoc_fetch(slot, out)
    return out


def test_maxmoc_windows_orca2():
    """One cell, one latitude, the whole (ny x nz) slab, every basin, and windows over the dry southern rows (a +0
    plateau: ties everywhere)."""
    m = synth.make_mesh("ORCA2")
    ib, e3m = case_inputs(oracle, m, synth)
    psi = moc_slab(m.e1v, e3m, ib, synth.make_v_record(m, 50)[:-1], slot=1)
    assert np.all(psi[:, 0] == 0.0)
    for basin in range(5):
        for win in ((1, m.ny, 1, m.nz), (40, 40, 12, 12), (70, 70, 1, m.nz), (1, 3, 1, m.nz), (1, 1, 5, 9),
                    (20, 120, 2, 20)):
            check_max(1, psi, basin, win)
    got = check_max(1, psi, 0, (1, 1, 1, m.nz))              # the closed southern row: psi = +0 everywhere
    assert got[0] == got[1] == 0.0 and got[2] == got[3] == (1, 1)


def test_maxmoc_ties():
    """Rows j and j + 7 identical (metrics, masks, V) and V non-zero at one level only: psi repeats exactly along the
    levels above it and between the two rows; the first cell in (j fastest, k) order wins."""
    m = synth.make_mesh("ODD")
    ib, e3m = case_inputs(oracle, m, synth)
    e1v, e3m, ib = m.e1v.copy(), e3m.copy(), ib.copy()
    v = np.zeros((m.nz - 1, m.ny, m.nx), F4)
    rng = np.random.default_rng(51)
    k = 2
    j = next(j for j in range(1, m.ny - 1) if (e3m[k, j] * ib[j, :, 0]).any())
    j2 = m.ny - 1
    e3m[:, j2], e1v[j2], ib[j2] = e3m[:, j], e1v[j], ib[j]
    v[k, j] = v[k, j2] = (0.1 * rng.standard_normal(m.nx)).astype(F4)
    psi = moc_slab(e1v, e3m, ib, v)
    assert psi[0, j, 0] == psi[k, j, 0] == psi[0, j2, 0] != 0.0
    for basin in range(5):
        got = check_max(0, psi, basin, (1, m.ny, 1, m.nz))
    got = check_max(0, psi, 0, (j + 1, m.ny, 1, m.nz))
    assert (got[2] if psi[0, j, 0] > 0 else got[3]) == (j + 1, 1)


def test_maxmoc_nonfinite_windows():
    """A NaN V cell poisons psi at its latitude for its level and every level above (cdfmoc does not scrub V): a window of
    one latitude there is all NaN; wider ones hold a few NaN cells.  +Inf V in a cell covered by a basin gives psi = -Inf
    there, -Inf gives +Inf; basins whose mask is 0 at that cell get 0 * Inf = NaN."""
    m = synth.make_mesh("ORCA2")
    ib, e3m = case_inputs(oracle, m, synth)
    v = synth.make_v_record(m, 52)[:-1].copy()
    kk = 9
    wet = lambda j: int(np.flatnonzero(e3m[kk, j] * ib[j, :, 0])[0])
    rows = [j for j in range(20, m.ny - 20) if (e3m[kk, j] * ib[j, :, 0]).any()]
    jn, jp, jm = rows[len(rows) // 4], rows[len(rows) // 2], rows[3 * len(rows) // 4]
    v[kk, jn, wet(jn)] = np.nan
    v[kk, jp, wet(jp)] = np.inf
    v[kk, jm, wet(jm)] = -np.inf
    with np.errstate(all="ignore"):
        psi = moc_slab(m.e1v, e3m, ib, v, slot=2)
    assert np.isnan(psi[: kk + 1, jn]).all() and np.isneginf(psi[: kk + 1, jp, 0]).all()
    wins = [(jn + 1, jn + 1, 1, kk + 1), (jn + 1, jn + 1, 3, 5), (jn - 5, jn + 5, 1, m.nz), (jp + 1, jp + 1, 1, kk + 1),
            (jm + 1, jm + 1, 1, kk + 1), (jp - 2, jm + 2, 1, m.nz), (1, m.ny, 1, m.nz), (jn + 1, jn + 1, 1, m.nz)]
    for basin in range(5):
        for win in wins:
            check_max(2, psi, basin, win)
    got = lib.cdfmoc_maxmoc(2, 0, jn + 1, jn + 1, 1, kk + 1)
    assert np.isnan(got[0]) and np.isnan(got[1]) and got[2] == got[3] == (jn + 1, 1)
    got = lib.cdfmoc_maxmoc(2, 0, jp + 1, jp + 1, 1, kk + 1)
    assert got[0] == got[1] == -np.inf and got[2] == got[3] == (jp + 1, 1)
    got = lib.cdfmoc_maxmoc(2, 0, jm + 1, jm + 1, 1, kk + 1)
    assert got[0] == got[1] == np.inf and got[2] == got[3] == (jm + 1, 1)


def test_maxmoc_full_window_orca025(orca025):
    """76 575 cells in one window: many per thread of the 256-thread block."""
    m = orca025
    ib, e3m = case_inputs(oracle, m, synth)
    psi = moc_slab(m.e1v, e3m, ib, synth.make_v_record(m, 53)[:-1])
    for basin in range(5):
        check_max(0, psi, basin, (1, m.ny, 1, m.nz))
    check_max(0, psi, 1, (600, 900, 10, 60))


def test_maxmoc_slots_and_errors():
    """Each slot's own slab; CDFGPU_ERR_ARG for an empty or out-of-range window or basin, CDFGPU_ERR_STATE for a slot
    nothing was submitted on."""
    m = synth.make_mesh("ODD")
    ib, e3m = case_inputs(oracle, m, synth)
    nz, ny, nb = lib.cdfmoc_setup(m.e1v, e3m, ib)
    psis = []
    for slot in range(3):
        out = np.empty((nz, ny, nb))
        lib.cdfmoc_submit(slot, slot, synth.make_v_record(m, 54 + slot)[:-1])
        lib.cdfmoc_fetch(slot, out)
        psis.append(out)
    for slot in (2, 1, 0):
        for basin in range(nb):
            check_max(slot, psis[slot], basin, (1, ny, 1, nz))
    lib.cdfmoc_setup(m.e1v, e3m, ib)
    lib.cdfmoc_submit(0, 0, synth.make_v_record(m, 54)[:-1])
    lib.cdfmoc_fetch(0, np.empty((nz, ny, nb)))
    for args, code in (((0, 0, 5, 4, 1, nz), ERR_ARG), ((0, 0, 1, ny, 3, 2), ERR_ARG), ((0, 0, 0, ny, 1, nz), ERR_ARG),
                       ((0, 0, 1, ny + 1, 1, nz), ERR_ARG), ((0, 0, 1, ny, 1, nz + 1), ERR_ARG), ((0, nb, 1, ny, 1, nz), ERR_ARG),
                       ((0, -1, 1, ny, 1, nz), ERR_ARG), ((1, 0, 1, ny, 1, nz), ERR_STATE)):
        with pytest.raises(lib.CdfGpuError) as e:
            lib.cdfmoc_maxmoc(*args)
        assert e.value.code == code, args
