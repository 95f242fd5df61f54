"""Shared helpers of the parity tests."""
import numpy as np

from cdftools_b200 import ncfiles

# north_star tolerance for the streamfunction: 1e-9 relative OR 1e-6 Sv absolute (fp64 summation order only)
RTOL_PSI = 1e-9
ATOL_PSI_SV = 1e-6


def assert_psi_close(got, ref, what=""):
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    nan_g, nan_r = np.isnan(got), np.isnan(ref)
    assert np.array_equal(nan_g, nan_r), f"{what}: NaN pattern differs ({nan_g.sum()} vs {nan_r.sum()})"
    inf_r = np.isinf(ref)
    assert np.array_equal(got[inf_r], ref[inf_r]), f"{what}: Inf pattern differs"
    ok = ~(nan_r | inf_r)
    err = np.abs(got[ok] - ref[ok])
    tol = np.maximum(RTOL_PSI * np.abs(ref[ok]), ATOL_PSI_SV)
    bad = err > tol
    assert not bad.any(), f"{what}: {bad.sum()} values out of tolerance, max abs err {err.max():.3e} Sv"
    return float(err.max()) if err.size else 0.0


def smem_bytes(iso, warps, nbins, npat1, nb, tab_rows=8):
    """sig_smem_bytes (api_mocsig.inc): what one CTA of K2 needs."""
    nh = 3 if iso else 1
    doubles = (warps * (nh * nbins * npat1 + tab_rows * 32) + nbins * nb + (nbins + 1) // 2 + 1) & ~1
    return doubles * 8 + 4 * warps * 32 * 16


# K2's shared-memory budget per CTA (sig_plan_units, api_mocsig.inc)
BUDGET = 227 * 1024 - 2048


def case_inputs(oracle, mesh, synth, with_basins=True, zero_edges=True):
    ib = oracle.basin_masks(*synth.basin_mask_inputs(mesh, with_basins), zero_edges=zero_edges)
    e3m = oracle.mask_e3v(mesh.e3v_0, mesh.vmask.astype(np.float32))
    return ib, e3m


def sigtrp_expected(oracle_mod, m, u, v, t, s, sec, smin, smax, nbins, spval=0.0, **kw):
    """What cdfsigtrp computes for one section from the arrays the files hold (src/cdfsigtrp.f90:404-627)."""
    imin, imax, jmin, jmax = sec
    e3w_1d, e3w = ncfiles.e3w_fields(m)
    e2u = (m.e1u * np.float32(0.9)).astype(np.float32)
    e3u = (m.e3v_0 * np.float32(1.01)).astype(np.float32)
    if imin == imax:   # meridional: rows jmin+1 .. jmax at column imin, T / S also at imin+1
        rows, i0 = slice(jmin, jmax), imin - 1
        cut = lambda a, i: np.ascontiguousarray(a[:, rows, i])
        eu, de3 = e2u[rows, i0].copy(), cut(e3u, i0)
        raw = dict(e3w_a=cut(e3w, i0), e3w_b=cut(e3w, i0 + 1), zu=cut(u, i0), zs_a=cut(s, i0), zs_b=cut(s, i0 + 1), zt_a=cut(t, i0),
                   zt_b=cut(t, i0 + 1))
        merid = True
    else:              # zonal: columns imin+1 .. imax at row jmin, T / S also at jmin+1; e1v starts at imin (as the reference reads it)
        cols, j0 = slice(imin, imax), jmin - 1
        cut = lambda a, j: np.ascontiguousarray(a[:, j, cols])
        eu, de3 = m.e1v[j0, imin - 1:imax - 1].copy(), cut(m.e3v_0, j0)
        raw = dict(e3w_a=cut(e3w, j0), e3w_b=cut(e3w, j0 + 1), zu=cut(v, j0), zs_a=cut(s, j0), zs_b=cut(s, j0 + 1), zt_a=cut(t, j0),
                   zt_b=cut(t, j0 + 1))
        merid = False
    p = oracle_mod.sigtrp_prepare(m.gdept_1d[0], raw["e3w_a"], raw["e3w_b"], raw["zu"], spval, raw["zs_a"], raw["zs_b"], spval, raw["zt_a"],
                                  raw["zt_b"], merid=merid)
    o = oracle_mod.sigtrp_section(eu, de3, p["ddepu"], m.gdepw_1d.astype(np.float32), p["zu"], p["zt"], p["zs"], p["zmask"], p["nk"], smin,
                                  smax, nbins, **kw)
    return p, o
