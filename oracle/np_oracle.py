"""Independent NumPy restatement of the cdfmoc / cdfmocsig hot path (TEST INFRASTRUCTURE ONLY).

Second, differently-structured restatement of the same reference loops as oracle/cdf_oracle.c.  It exists so
that the C oracle is checked by something that shares no code with it: the polynomial EOS is evaluated here
from the (i,j,k) coefficient table by a generic nested-Horner routine (the C file spells the expression out),
and the zonal sums use sequential ``np.cumsum`` prefix sums.  The two must agree bit for bit
(tests/test_oracle_cross.py).  Nothing in the product path imports this module.

Array conventions: C-order ``[k][j][i]`` (== Fortran ``(i,j,k)``), masks ``[j][i][b]`` int16,
``dmoc`` cdfmoc ``[k][j][b]`` float64, cdfmocsig ``[j][bin][b]`` float64.

Reference lines: src/cdfmoc.f90:325-336,352-388,520-551,590-594; src/cdfmocsig.f90:265-304,374-475;
src/eos.f90:207-279,408-466,661-684,842-882.
"""
from __future__ import annotations

import re
from pathlib import Path

import numpy as np

_HDR = Path(__file__).resolve().parent.parent / "include" / "cdf_eos_coeffs.h"


def _load_coeffs():
    txt = _HDR.read_text()
    tabs = {}
    for name in ("EOS80", "TEOS10"):
        body = txt.split("CDF_%s_COEF[CDF_EOS_NCOEF] = {" % name)[1].split("};")[0]
        d = {}
        for m in re.finditer(r"([-+0-9.eE]+),\s*/\*\s*EOS(\d)(\d)(\d)\s*\*/", body):
            d[(int(m.group(2)), int(m.group(3)), int(m.group(4)))] = float(m.group(1))
        tabs[name] = d
    r0 = [float(x) for x in txt.split("CDF_EOS_R0[6] = {")[1].split("}")[0].split(",")]
    return tabs, r0


_COEF, _R0 = _load_coeffs()
_PARAMS = {"EOS80": (20.0, 1.0 / 40.0), "TEOS10": (32.0, 0.875 / 35.16504)}


def _poly_k(E, k, t, s):
    """One of dlr0..dlr3 (eos.f90:858-877) with the reference's association:
    acc = E[0,J,k];  for j=J-1..0:  acc = (acc*t + Q_j) + E[0,j,k],  Q_j = (((E[I]*s+E[I-1])*s ...+E[1])*s."""
    js = sorted({j for (i, j, kk) in E if kk == k})
    J = js[-1]
    acc = np.full_like(t, E[(0, J, k)])
    for j in range(J - 1, -1, -1):
        I = max(i for (i, jj, kk) in E if kk == k and jj == j)
        q = np.full_like(s, E[(I, j, k)])
        for i in range(I - 1, 0, -1):
            q = q * s + E[(i, j, k)]
        q = q * s
        acc = (acc * t + q) + E[(0, j, k)]
    return acc


def eos_dlr(t32, s32, depth32, teos10=False):
    E = _COEF["TEOS10" if teos10 else "EOS80"]
    rdeltaS, r1_S0 = _PARAMS["TEOS10" if teos10 else "EOS80"]
    t = np.asarray(t32, np.float32).astype(np.float64) * (1.0 / 40.0)
    s = np.sqrt(np.abs(np.asarray(s32, np.float32).astype(np.float64) + rdeltaS) * r1_S0)
    h = np.float64(np.float32(depth32)) * 1.0e-4
    r3, r2, r1, r0 = (_poly_k(E, k, t, s) for k in (3, 2, 1, 0))
    return ((r3 * h + r2) * h + r1) * h + r0


def sigmai_dep(t32, s32, pref32, teos10=False):
    """eos.f90:842-882."""
    h = np.float64(np.float32(pref32)) * 1.0e-4
    R = _R0
    dlref = (((((R[5] * h + R[4]) * h + R[3]) * h + R[2]) * h + R[1]) * h + R[0]) * h
    dlr = eos_dlr(t32, s32, pref32, teos10)
    dltm = np.where(np.asarray(s32, np.float32) == np.float32(0), 0.0, 1.0)
    return (dlr + dlref - 1000.0) * dltm


def sigmantr(t32, s32):
    """eos.f90:661-684."""
    t = np.asarray(t32, np.float32).astype(np.float64)
    s = np.asarray(s32, np.float32).astype(np.float64)
    sr = np.sqrt(np.abs(s))
    r1 = ((-4.3159255086706703e-4 * t + 8.1157118782170051e-2) * t + 2.2280832068441331e-1) * t + 1002.3063688892480
    r2 = (-1.7052298331414675e-7 * s - 3.1710675488863952e-3 * t - 1.0304537539692924e-4) * s
    r3 = (((-2.3850178558212048e-9 * t - 1.6212552470310961e-7) * t + 7.8717799560577725e-5) * t
          + 4.3907692647825900e-5) * t + 1.0
    r4 = ((-2.2744455733317707e-9 * t * t + 6.0399864718597388e-6) * t - 5.1268124398160734e-4) * s
    r5 = (-1.3409379420216683e-9 * t * t - 3.6138532339703262e-5) * s * sr
    return (r1 + r2) / (r3 + r4 + r5) - 1000.0


def basin_masks(vmask1, atl=None, ind=None, pac=None, zero_edges=True):
    """cdfmoc.f90:325-336.  Inputs REAL(4) (ny,nx); returns int16 (ny,nx,nb)."""
    ny, nx = vmask1.shape
    nb = 5 if atl is not None else 1
    m = np.zeros((ny, nx, nb), np.int16)
    m[:, :, 0] = np.trunc(vmask1).astype(np.int16)
    if nb == 5:
        m[:, :, 1] = np.trunc(atl).astype(np.int16)
        m[:, :, 3] = np.trunc(ind).astype(np.int16)
        m[:, :, 4] = np.trunc(pac).astype(np.int16)
        ssum = (m[:, :, 4] + m[:, :, 3]).astype(np.int16)
        m[:, :, 2] = np.where(ssum > 0, np.int16(1), ssum)
    if zero_edges:
        m[:, 0, 0] = 0
        m[:, nx - 1, 0] = 0
    return m


def mask_e3v(e3v_file, vmask):
    """cdfmoc.f90:590-594."""
    return (e3v_file.astype(np.float32) * np.trunc(vmask).astype(np.int16).astype(np.float32)).astype(np.float32)


def cdfmoc_record(e1v, e3m, ibmask, zv):
    """cdfmoc.f90:352-388.  e1v (ny,nx) f32; e3m (nz,ny,nx) f32; ibmask (ny,nx,nb) i16; zv (nz-1,ny,nx) f32.
    Returns dmoc (nz,ny,nb) f64 (scanned, Sv)."""
    nz, ny, nx = e3m.shape
    nb = ibmask.shape[2]
    dmoc = np.zeros((nz, ny, nb), np.float64)
    mf = ibmask.astype(np.float32)
    for k in range(nz - 1):
        a = (e1v * e3m[k]).astype(np.float32)
        for b in range(nb):
            t = ((a * mf[:, :, b]).astype(np.float32) * zv[k]).astype(np.float32)
            # 0 - t0 - t1 - ... == -(t0 + t1 + ...) bit for bit (round-to-nearest is sign-symmetric)
            dmoc[k, :, b] = -np.cumsum(t.astype(np.float64), axis=1)[:, -1]
    dmoc = dmoc + 0.0  # normalise -0.0
    for k in range(nz - 2, -1, -1):
        dmoc[k] = dmoc[k + 1] + dmoc[k] / 1.0e6
    return dmoc


def cdfmoc_output(dmoc):
    """cdfmoc.f90:520-551 -> (nvar, nz, ny) f32, inp0 last when nb==5."""
    nz, ny, nb = dmoc.shape
    outs = [dmoc[:, :, b].astype(np.float32) for b in range(nb)]
    if nb >= 5:
        outs.append((dmoc[:, :, 0] - dmoc[:, :, 1]).astype(np.float32))
    return np.stack(outs)


def sigma_axis(nbins, sigmin, sigstp):
    """cdfmocsig.f90:302-304 in REAL(4)."""
    n = np.arange(1, nbins + 1, dtype=np.float32)
    return (np.float32(sigmin) + ((n - np.float32(0.5)) * np.float32(sigstp)).astype(np.float32)).astype(np.float32)


def mocsig_bins(zt, zs, zsps, pref, eos, sigmin, sigstp, nbins):
    """cdfmocsig.f90:393-403 on already-scrubbed zt, zs.  eos: 0 EOS80, 1 TEOS10, 2 neutral."""
    itmask = np.where(zs == np.float32(zsps), 0, 1).astype(np.int16)
    dens = sigmantr(zt, zs) if eos == 2 else sigmai_dep(zt, zs, pref, teos10=(eos == 1))
    zttmp = (dens * itmask.astype(np.float64)).astype(np.float32)
    q = ((zttmp - np.float32(sigmin)).astype(np.float32) / np.float32(sigstp)).astype(np.float32)
    # INT(): truncation toward zero; out of range and NaN give INT_MIN (x86 CVTTSS2SI, what gfortran emits), as cdf_oracle.c
    inr = (q > np.float32(-2147483648.0)) & (q < np.float32(2147483648.0))
    ib = np.where(inr, np.trunc(np.where(inr, q, np.float32(0))), -2147483648.0).astype(np.int64)
    ib = np.minimum(np.maximum(ib, 1), nbins).astype(np.int32)
    return ib, itmask, dens


def cdfmocsig_record(e1v, e3v, ibmask, zv, zt, zs, spv, spt, sps, pref, eos, sigmin, sigstp, nbins, zveiv=None):
    """cdfmocsig.f90:366-475.  Returns (dmoc (ny,nbins,nb) f64 scanned, ibin (nz-1,ny,nx) int32)."""
    nzm1, ny, nx = zv.shape
    nb = ibmask.shape[2]
    H = np.zeros((ny, nbins, nb), np.float64)
    bins = np.zeros((nzm1, ny, nx), np.int32)
    j1, j2 = (1, ny - 2) if ny > 1 else (0, 0)
    for k in range(nzm1):
        v = np.where(zv[k] == np.float32(spv), np.float32(0), zv[k]).astype(np.float32)
        if zveiv is not None:
            v = (v + zveiv[k]).astype(np.float32)
        t = np.where(zt[k] == np.float32(spt), np.float32(0), zt[k]).astype(np.float32)
        s = np.where(zs[k] == np.float32(sps), np.float32(0), zs[k]).astype(np.float32)
        area = (e1v * e3v[k]).astype(np.float32)
        ib, _, _ = mocsig_bins(t, s, sps, pref, eos, sigmin, sigstp, nbins)
        bins[k] = ib
        p = (v * area).astype(np.float32)
        contrib = 0.0 - p.astype(np.float64)
        for j in range(j1, j2 + 1):
            for i in range(1, nx - 1):  # sequential, i ascending: the order the reference sums in
                H[j, ib[j, i] - 1, :] += contrib[j, i] * ibmask[j, i, :].astype(np.float64)
    H[:, nbins - 1, :] = H[:, nbins - 1, :] / 1.0e6
    for b in range(nbins - 2, -1, -1):
        H[:, b, :] = H[:, b + 1, :] + H[:, b, :] / 1.0e6
    return H, bins


def isodep_record(e1v, e3v, ibmask, gdept, zt, zs, spt, sps, pref, eos, sigmin, sigstp, nbins):
    """cdfmocsig.f90:423-430,444-454,463-469 -> depi (ny,nbins,nb) f64 (mean isopycnal depth, 99999. where empty)."""
    nzm1, ny, nx = zt.shape
    nb = ibmask.shape[2]
    D = np.zeros((ny, nbins, nb)); W = np.zeros((ny, nbins, nb))
    j1, j2 = (1, ny - 2) if ny > 1 else (0, 0)
    for k in range(nzm1):
        t = np.where(zt[k] == np.float32(spt), np.float32(0), zt[k]).astype(np.float32)
        s = np.where(zs[k] == np.float32(sps), np.float32(0), zs[k]).astype(np.float32)
        area = (e1v * e3v[k]).astype(np.float32)
        ib, itm, _ = mocsig_bins(t, s, sps, pref, eos, sigmin, sigstp, nbins)
        gd = np.float32(-np.float32(gdept[k]))
        a = ((gd * itm.astype(np.float32)).astype(np.float32) * area).astype(np.float32).astype(np.float64)
        w = (itm.astype(np.float32) * area).astype(np.float32).astype(np.float64)
        for j in range(j1, j2 + 1):
            for i in range(1, nx - 1):
                D[j, ib[j, i] - 1, :] += a[j, i] * ibmask[j, i, :].astype(np.float64)
                W[j, ib[j, i] - 1, :] += w[j, i] * ibmask[j, i, :].astype(np.float64)
    with np.errstate(all="ignore"):
        return np.where(W != 0.0, D / np.where(W != 0.0, W, 1.0), 99999.0)


def _sinf(x32):
    """libm's sinf, element by element: the value the Fortran run-time's REAL(4) SIN gives on this platform."""
    import ctypes
    libm = ctypes.CDLL("libm.so.6")
    libm.sinf.restype, libm.sinf.argtypes = ctypes.c_float, [ctypes.c_float]
    flat = np.asarray(x32, np.float32).ravel()
    uniq, inv = np.unique(flat, return_inverse=True)
    vals = np.array([libm.sinf(float(u)) for u in uniq], np.float32)
    return vals[inv].reshape(np.shape(x32))


def cdfmoc_decomp_record(e1v, e1u, gphiv, gdept, e3m, ibmask, umask, tmask, zv, zt, zs, teos10=False):
    """cdfmoc -decomp, src/cdfmoc.f90:390-517 (vectorised restatement; zonal sums via sequential cumsum)."""
    f4, f8 = np.float32, np.float64
    nz, ny, nx = e3m.shape
    nb = ibmask.shape[2]
    mf = ibmask.astype(f4)
    total = cdfmoc_record(e1v, e3m, ibmask, zv)

    def weighted(dv):
        out = np.zeros((nz, ny, nb))
        for k in range(nz - 1):
            a = (e1v * e3m[k]).astype(f4)
            for b in range(nb):
                t = (a * mf[:, :, b]).astype(f4).astype(f8) * dv
                out[k, :, b] = -np.cumsum(t, axis=1)[:, -1]
        return out + 0.0

    def scan(d):
        d = d.copy()
        for k in range(nz - 2, -1, -1):
            d[k] = d[k + 1] + d[k] / 1.0e6
        return d

    dvbt = np.zeros((ny, nx)); hdep = np.zeros((ny, nx), f4)
    for k in range(nz - 1):
        dvbt = dvbt + (e3m[k] * zv[k]).astype(f4).astype(f8)
        hdep = (hdep + e3m[k]).astype(f4)
    with np.errstate(all="ignore"):
        dvbt = np.where(hdep != 0, dvbt / np.where(hdep != 0, hdep, 1).astype(f8), 0.0)
    bt = scan(weighted(dvbt))

    rpi = f4(np.arccos(f4(-1.0)))
    f = f4(f4(4.0) * rpi) / f4(f4(24.0) * f4(3600.0))
    ang = ((rpi * gphiv.astype(f4)).astype(f4) / f4(180.0)).astype(f4)
    fcor = (f4(f) * _sinf(ang)).astype(f4)
    g = f4(f4(-9.81) / f4(1025.0))
    with np.errstate(all="ignore"):
        zcoef = np.where(fcor != 0, (g / np.where(fcor != 0, fcor, 1)).astype(f4), f4(0)).astype(f4)

    dvgeo = np.zeros((2, ny, nx)); dvbt = np.zeros((ny, nx)); sh = np.zeros((nz, ny, nb))
    zvg = zv[nz - 2].astype(f4).copy()          # border cells keep the last level read by the first loop
    iup, ido = 0, 1
    J, I = slice(1, ny - 1), slice(1, nx - 1)
    for k in range(nz - 2, -1, -1):
        um = umask[k].astype(np.int16); umf = um.astype(f4)
        sig = (sigmai_dep(zt[k], zs[k], gdept[k], teos10) * tmask[k].astype(f8)).astype(f4)
        su = (um[2:, 0:-2] + um[2:, 1:-1] + um[1:-1, 0:-2] + um[1:-1, 1:-1]).astype(np.int16)
        zmsv = (f4(1.0) / np.maximum(su, 1).astype(f4)).astype(f4)
        def term(sa, sb, u, e):   # ((sa - sb) * real(u)) / e  in REAL(4)
            return (((sa - sb).astype(f4) * u).astype(f4) / e).astype(f4)
        t1 = term(sig[2:, 1:-1], sig[2:, 0:-2], umf[2:, 0:-2], e1u[2:, 0:-2])
        t2 = term(sig[2:, 2:], sig[2:, 1:-1], umf[2:, 1:-1], e1u[2:, 1:-1])
        t3 = term(sig[1:-1, 1:-1], sig[1:-1, 0:-2], umf[1:-1, 0:-2], e1u[1:-1, 0:-2])
        t4 = term(sig[1:-1, 2:], sig[1:-1, 1:-1], umf[1:-1, 1:-1], e1u[1:-1, 1:-1])
        dgeo = (((t1 + t2).astype(f4) + t3).astype(f4) + t4).astype(f4).astype(f8)
        d = zcoef[J, I].astype(f8) * dgeo
        d = d * zmsv.astype(f8)
        d = d * ibmask[J, I, 0].astype(f8)
        d = d * e3m[k][J, I].astype(f8)
        dvgeo[iup][J, I] = dvgeo[ido][J, I] + d
        zvg[J, I] = (0.5 * (dvgeo[iup][J, I] + dvgeo[ido][J, I])).astype(f4)
        dvbt = dvbt + (e3m[k] * zvg).astype(f4).astype(f8)
        a = (e1v * e3m[k]).astype(f4)
        for b in range(nb):
            t = ((a * mf[:, :, b]).astype(f4) * zvg).astype(f4)
            sh[k, :, b] = -np.cumsum(t.astype(f8), axis=1)[:, -1]
        iup, ido = ido, iup
    sh = sh + 0.0
    with np.errstate(all="ignore"):
        dvbt = np.where(hdep != 0, dvbt / np.where(hdep != 0, hdep, 1).astype(f8), 0.0)
    sh = scan(sh - weighted(dvbt))
    return {"total": total, "sh": sh, "bt": bt, "ag": total - sh - bt}


def maxmoc(rmoc, ijmin, ijmax, ikmin, ikmax):
    """cdfmaxmoc.f90:158-167 as gfortran's MAXVAL / MAXLOC (MINVAL / MINLOC) compute them on the REAL(4) window
    rmoc (nz, ny)[ikmin-1:ikmax, ijmin-1:ijmax]: NaN cells never count; the location is the first cell in (jj fastest,
    jk) order whose value equals the extremum; a window without a non-NaN cell gives NaN at its first cell.
    -> (ovtmax, ovtmin, (jj,jk) of max, (jj,jk) of min), 1-based."""
    w = np.asarray(rmoc, np.float32)[ikmin - 1:ikmax, ijmin - 1:ijmax]
    nj = w.shape[1]
    flat = w.ravel()                       # C order of [k][j]: jj fastest
    ok = ~np.isnan(flat)
    if not ok.any():
        return np.float32(np.nan), np.float32(np.nan), (ijmin, ikmin), (ijmin, ikmin)
    out = []
    for ext in (flat[ok].max(), flat[ok].min()):
        n = int(np.flatnonzero(ok & (flat == ext))[0])
        out.append((flat[n], (ijmin + n % nj, ikmin + n // nj)))
    return out[0][0], out[1][0], out[0][1], out[1][1]


# ---- sibling tools (SURVEY.md section 8 f3): independent NumPy restatements ----------------------------------------
f4, f8 = np.float32, np.float64

def zonalsum_record(zmask, zmaskvar, zv, e1, e2, alpha=None):
    """cdfzonalsum.f90:257,309-322.  zmask (ny,nx,nb) f32, zmaskvar / zv (nk,ny,nx) f32 -> (nb,nk,ny) f64."""
    dl = (f8(1.0) * e1.astype(f8)) * e2.astype(f8)
    nk, ny, nx = zv.shape
    nb = zmask.shape[2]
    out = np.empty((nb, nk, ny), f8)
    al = np.ones(ny, f4) if alpha is None else alpha.astype(f4)
    for b in range(nb):
        for k in range(nk):
            p = ((zmask[:, :, b] * zmaskvar[k]).astype(f4) * zv[k]).astype(f4).astype(f8)
            out[b, k] = np.cumsum(dl * p, axis=1)[:, -1] / al.astype(f8)   # cumsum: sequential in i like the DO loop
    return out


def zonalmean_record(zmask, zmaskvar, zv, e1, e2, zspval=0.0, lmax=False):
    """cdfzonalmean.f90:265,312-344 -> mean (nb,nk,ny) f64, zmax, zmin (nb,nk,ny) f32 (None without lmax)."""
    dl = (f8(1.0) * e1.astype(f8)) * e2.astype(f8)
    nk, ny, nx = zv.shape
    nb = zmask.shape[2]
    mean = np.empty((nb, nk, ny), f8)
    zmax = np.empty((nb, nk, ny), f4) if lmax else None
    zmin = np.empty((nb, nk, ny), f4) if lmax else None
    for b in range(nb):
        m = zmask[:, :, b].astype(f8)
        for k in range(nk):
            dtmp = ((f8(1.0) * m) * zmaskvar[k].astype(f8)) * zv[k].astype(f8)
            acc = np.cumsum(dl * dtmp, axis=1)[:, -1]
            area = np.cumsum((dl * m) * zmaskvar[k].astype(f8), axis=1)[:, -1]
            with np.errstate(all="ignore"):
                mean[b, k] = np.where(area != 0, acc / np.where(area != 0, area, 1.0), f8(f4(zspval)))
            if lmax:   # fmax / fmin: a NaN cell never changes the zonal max / min
                mx = np.fmax(f8(f4(-1.e20)), np.fmax.reduce(dtmp, axis=1)).astype(f4)
                mn = np.fmin(f8(f4(1.e20)), np.fmin.reduce(np.where(dtmp != 0, dtmp, np.inf), axis=1)).astype(f4)
                zmax[b, k] = np.where(area == 0, f4(zspval), mx)
                zmin[b, k] = np.where(area == 0, f4(zspval), mn)
    return mean, zmax, zmin


def mhst_record(e1v, e3v, vmask1, zvt, zvs, atl=None, pac=None, ind=None, zdim=False):
    """cdfmhst.f90:303-366 -> heat, salt (nlev,4,ny) f64 raw zonal sums, order glo, atl, pac, ind."""
    nz, ny, nx = zvt.shape
    nlev = nz if zdim else 1
    heat, salt = np.zeros((nlev, 4, ny), f8), np.zeros((nlev, 4, ny), f8)
    dtrph, dtrps = np.zeros((ny, nx), f8), np.zeros((ny, nx), f8)
    masks = [vmask1, atl, pac, ind]
    for k in range(nz):
        dwkh = ((zvt[k] * e1v).astype(f4) * e3v[k]).astype(f4).astype(f8)
        dwks = ((zvs[k] * e1v).astype(f4) * e3v[k]).astype(f4).astype(f8)
        dtrph = dtrph + (dwkh * f8(f4(1000.0))) * f8(f4(4000.0))
        dtrps = dtrps + dwks
        if zdim or k == nz - 1:
            lev = k if zdim else 0
            for m, mk in enumerate(masks):
                if mk is None:
                    continue
                sl = slice(1, nx - 1) if m == 0 else slice(0, nx)
                heat[lev, m] = np.cumsum(dtrph[:, sl] * mk[:, sl].astype(f8), axis=1)[:, -1]
                salt[lev, m] = np.cumsum(dtrps[:, sl] * mk[:, sl].astype(f8), axis=1)[:, -1]
    return heat, salt


# ---- cdftransig_xy3d (src/cdftransig_xy3d.f90) -------------------------------------------------------------------
def transig_bins(nbins, ds1min, ds1scal, ds1zoom=999.0, ds1scalmin=999.0):
    """Bin centres, edges and the step -> bin look-up table (:213, :229-262).  itab is 1-based, 0 = no bin."""
    ds1scalmin = min(ds1scalmin, ds1scal)
    ji = np.arange(1, nbins + 1)
    test = ds1min + (ji - 0.5) * ds1scal
    zoom = test > ds1zoom
    dsigma = test.copy()
    if zoom.any():
        ijtrans = int(ji[zoom][0])
        dsigma[zoom] = ds1zoom + (ji[zoom] - ijtrans + 0.5) * ds1scalmin
    edge = np.empty(nbins + 1)
    edge[0] = ds1min
    edge[1:nbins] = 0.5 * (dsigma[1:] + dsigma[:-1])
    edge[nbins] = edge[nbins - 1] + ds1scalmin
    x = (edge[nbins] - edge[0]) / ds1scalmin
    nsigmax = int(np.floor(abs(x) + 0.5) * np.sign(x))                       # NINT
    t = ds1min + (np.arange(1, nsigmax + 1) - 0.5) * ds1scalmin
    itab = np.zeros(nsigmax, np.int32)
    for jj in range(1, nbins + 1):                                           # the last bin that claims a step wins
        itab[(t > edge[jj - 1]) & (t <= edge[jj])] = jj
    return dsigma, edge, itab, ds1scalmin


def _int_d(x):
    """Fortran INT() of REAL(8) with x86 CVTTSD2SI semantics (out of range / NaN -> INT_MIN)."""
    bad = ~((x > -2147483649.0) & (x < 2147483648.0))
    r = np.trunc(np.where(bad, 0.0, x)).astype(np.int64)
    r[bad] = -2147483648
    return r


def transig_record(e2u, e1v, e3u, e3v, zu, zv, zt, zs, pref, ds1min, ds1scalmin, itab, nbins, dusig, dvsig, masku, maskv,
                   set_masks=True, lperio=False, teos10=False):
    """One frame, all levels (:396-461), accumulated in place into dusig / dvsig (nbins, ny, nx)."""
    f32 = np.float32
    nzm1, ny, nx = zu.shape
    nsigmax = itab.size
    jj, ii = np.meshgrid(np.arange(ny), np.arange(nx), indexing="ij")
    for k in range(nzm1):
        dens = sigmai_dep(zt[k], zs[k], f32(pref), teos10)
        if set_masks:
            masku[k] = (zu[k] != 0).astype(np.uint8)
            maskv[k] = (zv[k] != 0).astype(np.uint8)
        zdu = np.zeros((ny, nx), f32)
        zdu[:, :-1] = (0.5 * (dens[:, :-1] + dens[:, 1:])).astype(f32)
        if lperio and nx > 2:
            zdu[:, -1] = zdu[:, 1]
        zdu = zdu * masku[k].astype(f32)
        zdv = np.zeros((ny, nx), f32)
        zdv[:-1] = (0.5 * (dens[:-1] + dens[1:])).astype(f32)
        zdv = zdv * maskv[k].astype(f32)
        for zd, vel, e3, e12, acc in ((zdu, zu[k], e3u[k], e2u, dusig), (zdv, zv[k], e3v[k], e1v, dvsig)):
            ijb = np.clip(_int_d((zd.astype(np.float64) - ds1min) / ds1scalmin) + 1, 1, nsigmax)
            b = itab[ijb - 1]
            p = (e12.astype(f32) * (vel.astype(f32) * e3.astype(f32))).astype(np.float64) * 1.0
            ok = b >= 1
            acc[b[ok] - 1, jj[ok], ii[ok]] += p[ok]                          # one (bin, j, i) per cell: no duplicates


# ---- cdfsigtrp (src/cdfsigtrp.f90) ---------------------------------------------------------------------------------
def sigtrp_prepare(gdept1, e3w_a, e3w_b, zu, zspu, zs_a, zs_b, zsps, zt_a, zt_b, merid=False):
    """:428-460 / :521-555, vectorised over the section; arrays (npk, npts) float32."""
    f32 = np.float32
    npk, npts = zu.shape
    ddepu = np.zeros((npk + 1, npts), np.float64)
    ddepu[1] = np.float64(f32(gdept1))
    for k in range(1, npk):
        ddepu[k + 1] = ddepu[k] + np.minimum(e3w_a[k], e3w_b[k]).astype(np.float64)
    zu = np.where(zu == f32(zspu), f32(0), zu).astype(f32)
    zmask = np.where((zs_a == f32(zsps)) | (zs_b == f32(zsps)), f32(0), f32(1)).astype(f32)
    zs = (f32(0.5) * (zs_a + zs_b)) * zmask
    zt = f32(0.5) * (zt_a + zt_b)
    if merid:
        zt = zt * zmask
    nk, found = npk, False
    for k in range(npk):
        s = f32(0)
        for v in zs[k]:
            s = f32(s + v)
        if s == 0:
            nk, found = k + 1, True
            break
    return dict(ddepu=ddepu, zu=zu, zs=zs.astype(f32), zt=zt.astype(f32), zmask=zmask, nk=nk, found=found)


def sigtrp_section(eu, de3, ddepu, gdepw, zu, zt, zs, zmask, nk, dsigma_min, dsigma_max, nbins, mode=0, refdep=0.0,
                   teos10=False, ddepw_brk=None):
    """:559-627, vectorised over the section, explicit loops over levels and class limits."""
    f64 = np.float64
    npk, npts = zu.shape
    lev = np.empty(nbins + 1, f64)
    dlt = (f64(dsigma_max) - f64(dsigma_min)) / f64(nbins)
    lev[0] = dsigma_min
    for c in range(2, nbins + 2):
        lev[c - 1] = lev[0] + f64(c - 1) * dlt
    dsig = np.zeros((nk + 1, npts), f64)
    if mode == 2:
        dsig[1:] = ((-zt[:nk]) * zmask[:nk]).astype(f64)
    else:
        d = sigmantr(zt[:nk], zs[:nk]) if mode == 1 else sigmai_dep(zt[:nk], zs[:nk], np.float32(refdep), teos10)
        dsig[1:] = d * zmask[:nk].astype(f64)
    dsig[0] = dsig[1] - f64(np.float32(1.e-4))
    for k in range(1, nk + 1):
        land = zmask[k - 1] == 0
        dsig[k] = np.where(land, dsig[k - 1] + f64(np.float32(1.e-5)), dsig[k])
    dhiso = np.empty((nbins + 1, npts), f64)
    dwtrp = np.empty((nbins + 1, npts), f64)
    e = eu.astype(f64)
    with np.errstate(all="ignore"):
        for iso in range(nbins + 1):
            h = ddepu[npk].copy()
            done = np.zeros(npts, bool)
            for k in range(1, nk + 1):
                hit = ~done & ~(dsig[k] < lev[iso])
                if hit.any():
                    dalfa = (lev[iso] - dsig[k - 1]) / (dsig[k] - dsig[k - 1])
                    val = ddepu[k] * dalfa + (1.0 - dalfa) * ddepu[k - 1]
                    val = np.where((np.abs(dalfa) > 1.1) | (dalfa < 0.0), 0.0, val)
                    h = np.where(hit, val, h)
                    done |= hit
            dhiso[iso] = h
            w = np.zeros(npts, f64)
            done = np.zeros(npts, bool)
            for k in range(1, nk):
                gw1 = (ddepw_brk[k] if ddepw_brk is not None else np.full(npts, gdepw[k], np.float32)).astype(f64)
                gw0 = (ddepw_brk[k - 1] if ddepw_brk is not None else np.full(npts, gdepw[k - 1], np.float32)).astype(f64)
                u = zu[k - 1].astype(f64)
                full = gw1 < h
                add = np.where(full, (e * de3[k - 1].astype(f64)) * u, (e * (h - gw0)) * u)
                w = np.where(done, w, w + add)
                done |= ~full
            dwtrp[iso] = w
    dwtrpbin = dwtrp[1:] - dwtrp[:-1]
    dtrpbin = np.empty(nbins, f64)
    for b in range(nbins):
        s = f64(0)
        for v in dwtrpbin[b]:
            s = s + v
        dtrpbin[b] = s
    return dict(dsigma_lev=lev, dsig=dsig, dhiso=dhiso, dwtrp=dwtrp, dwtrpbin=dwtrpbin, dtrpbin=dtrpbin)
