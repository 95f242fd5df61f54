"""The sibling kernels against the C oracle at production widths and at the shapes where their indexing changes:
K4 zonal_rows_kernel (cdfzonalsum / cdfzonalmean), K5 mhst_rows_kernel and K5v mhst_vpoint_kernel (cdfmhst), K6
transig_scatter_kernel (cdftransig_xy3d).

Two kinds of reference:
  * exact inputs -- metrics that are powers of two, data that are small integers times powers of two, each value derived
    from the cell's flat (k, j, i) index.  Every product and every partial sum is then exact, so any order of additions
    gives the same bits: the kernel must equal the C oracle bit for bit, and a dropped, repeated or misplaced cell shows.
  * random inputs -- the per-cell terms formed in the reference's own fp32 / fp64 chain and summed row by row with
    math.fsum (correctly rounded).  A kernel sum whose longest chain of fp64 additions is D is within
    gamma_D * sum|terms| of the exact sum (gamma_D = D u / (1 - D u), u = 2^-53); the checks allow twice that.
    The sequential oracle's own error at nx = 8192 is as large as 1e-12 relative, so it is not the reference here.
K6 adds into each accumulator in the oracle's order (frame, then level; one thread per column): bit for bit always."""
import math

import numpy as np
import pytest

import oracle
from cdftools_b200 import lib, synth
from test_gpu_sibling_inputs import vpoint
from test_transig import CODES

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
ZSP = -99999.0          # zspval: the fill of rows without area
ERR_ARG = 2             # CDFGPU_ERR_ARG


@pytest.fixture(scope="module", autouse=True)
def _ctx(gpu_lib, oracle_mod):
    """The session-wide library context (conftest.gpu_lib), never finalised here: the test modules that follow use it."""
    yield


def gamma(d):
    return d * U / (1.0 - d * U)


def same_bits(a, b):
    """Equal bit for bit (so +0 differs from -0); a NaN equals a NaN whatever its payload."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    it = {8: np.int64, 4: np.int32}[a.dtype.itemsize]
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(it), b[~nb].view(it))


def same_values(a, b):
    """Zonal max / min: equal values.  Which zero a row's max of +0 and -0 cells keeps depends on the order of the
    comparisons in the reference too, so the sign of a zero is not compared."""
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


def exact_field(shape, nbits=12, offset=0):
    """Small integers (< 2^nbits) times 2^0..2^-4, signs mixed, each value a function of the cell's flat index."""
    code = np.arange(int(np.prod(shape)), dtype=np.int64).reshape(shape) + offset
    mag = code % ((1 << nbits) - 3) + 1
    sgn = np.where(code % 3 == 0, -1.0, 1.0)
    return (sgn * mag * 2.0 ** -(code % 5)).astype(np.float32)


def pow2(rng, shape):
    return (2.0 ** rng.integers(-1, 2, shape)).astype(np.float32)


# ---- K4: cdfzonalsum / cdfzonalmean -------------------------------------------------------------------------------------
def zonal_exact(nx, ny, nk, nb, seed, general=None):
    """-> e1, e2, zmask (ny,nx,nb), zmaskvar, zv, alpha.  general: one mask value (0.5 or -0.0) that sends K4 down
    the unpacked path (zonal_rows_kernel<NB, *, false>).  Row (k=0, j=0) and basin 0 of the last row have no area."""
    rng = np.random.default_rng(seed)
    e1, e2 = pow2(rng, (ny, nx)), pow2(rng, (ny, nx))
    mv = (rng.random((nk, ny, nx)) > 0.2).astype(np.float32)
    zm = (rng.random((ny, nx, nb)) > 0.4).astype(np.float32)
    mv[0, 0, :] = 0.0
    zm[ny - 1, :, 0] = 0.0
    if general is not None:
        zm[ny // 2, nx // 2, nb - 1] = general
    alpha = pow2(rng, ny) * np.float32(1.5)
    return e1, e2, zm, mv, exact_field((nk, ny, nx)), alpha


def check_zonal(e1, e2, zm, mv, zvs, alpha):
    """K4 sum (alpha and NULL), mean, mean with lmax on each record of zvs, all bit for bit against the C oracle."""
    dl = oracle.zonal_dlsurf(e1, e2)
    shape = lib.cdfzonal_setup(e1, e2, zm, mv)
    try:
        for n, zv in enumerate(zvs):
            for al in (alpha, None):
                got, ref = lib.cdfzonal_sum(zv, shape, al), oracle.zonalsum_record(zm, mv, zv, dl, al)
                assert same_bits(got, ref), f"record {n}: sum, alpha {al is not None}"
            for lmax in (False, True):
                got, ref = lib.cdfzonal_mean(zv, shape, ZSP, lmax), oracle.zonalmean_record(zm, mv, zv, dl, ZSP, lmax)
                assert same_bits(got[0], ref[0]), f"record {n}: mean, lmax {lmax}"
                if lmax:
                    assert same_values(got[1], ref[1]), f"record {n}: max"
                    assert same_values(got[2], ref[2]), f"record {n}: min"
                    empty = ref[0] == ZSP
                    assert np.all(got[1][empty] == np.float32(ZSP)) and np.all(got[2][empty] == np.float32(ZSP))
    finally:
        lib.cdfzonal_teardown()
    return ref


@pytest.mark.parametrize("general", [None, 0.5, -0.0], ids=["bits", "half", "negzero"])
@pytest.mark.parametrize("nx", [1, 2, 3, 4, 5, 7, 31, 33, 129, 1442, 4322])
def test_k4_widths(nx, general):
    """6 rows: with odd nx the 16-byte misalignment e0 & 3 of a row start takes all four values."""
    e1, e2, zm, mv, zv, alpha = zonal_exact(nx, 3, 2, 3, nx, general)
    ref = check_zonal(e1, e2, zm, mv, [zv], alpha)
    assert np.all(ref[0][:, 0, 0] == ZSP) and np.all(ref[0][0, :, -1] == ZSP)   # the rows without area were there


@pytest.mark.parametrize("general", [None, 0.5], ids=["bits", "half"])
@pytest.mark.parametrize("nb", range(1, 9))
def test_k4_basin_counts(nb, general):
    check_zonal(*_split(zonal_exact(37, 5, 3, nb, 100 + nb, general)))


def _split(case):
    e1, e2, zm, mv, zv, alpha = case
    return e1, e2, zm, mv, [zv], alpha


@pytest.mark.parametrize("general", [None, -0.0], ids=["bits", "negzero"])
@pytest.mark.parametrize("shape", [(33, 1, 4), (33, 4, 1), (1, 1, 1), (4, 1, 1), (7, 1500, 8)],
                         ids=["ny1", "nk1", "one-cell", "one-vector", "12000-rows"])
def test_k4_edge_shapes(shape, general):
    """ny = 1, nk = 1, a single cell, and (7, 1500, 8): 12000 (k, j) rows, more than one pass of the grid-stride loop
    (min(rows / 8, SMs * 8) blocks of 8 warps cover 9472 rows a pass on a B200)."""
    nx, ny, nk = shape
    check_zonal(*_split(zonal_exact(nx, ny, nk, 5, nx * ny + nk, general)))


def _row_parts(nx, ny, k, j):
    """Head (scalar cells before the first 16-byte boundary), vector body and tail of row (k, j) as K4 splits it."""
    e0 = (k * ny + j) * nx
    head = min((4 - e0 % 4) % 4, nx)
    nvec = (nx - head) // 4
    return head, nvec, nx - head - 4 * nvec


def test_k4_nonfinite_cell_in_head_body_and_tail():
    """A non-finite cell where the basin masks are mixed: the reference's mask-0 term is 0 * Inf = NaN, which the fast
    form of K4 (DFMA with a 1.0 / 0.0 multiplier) does not produce; the warp must redo the row with the literal chain
    wherever in the row the cell is.  One record per position."""
    nx, ny, nk, nb = 33, 5, 3, 3
    e1, e2, zm, mv, zv, alpha = zonal_exact(nx, ny, nk, nb, 7)
    k, j = next((k, j) for k in range(nk) for j in range(1, ny - 1)
                if _row_parts(nx, ny, k, j)[0] > 0 and _row_parts(nx, ny, k, j)[2] > 0)
    head, nvec, tail = _row_parts(nx, ny, k, j)
    recs = []
    for i, bad in ((0, np.inf), (head + 4 * (nvec // 2) + 1, np.nan), (nx - 1, -np.inf)):
        zm[j, i] = [1.0, 0.0, 1.0]
        mv[k, j, i] = 1.0
        z = zv.copy()
        z[k, j, i] = bad
        recs.append(z)
    check_zonal(e1, e2, zm, mv, recs, alpha)
    dl = oracle.zonal_dlsurf(e1, e2)
    for z in recs:   # the references are what the test means: the row is non-finite in every basin, the others finite
        ref = oracle.zonalsum_record(zm, mv, z, dl)
        assert not np.isfinite(ref[:, k, j]).any() and np.isnan(ref[1, k, j])
        assert np.isfinite(np.delete(ref.reshape(nb, -1), k * ny + j, axis=1)).all()


@pytest.mark.parametrize("general", [None, 0.5], ids=["bits", "half"])
def test_k4_nan_cells_under_lmax(general):
    """cdfzonalmean -max with NaN cells (include/cdfgpu.h): a NaN never changes the zonal max / min, the mean is NaN,
    a row whose every cell is NaN keeps -1.e20 / 1.e20; rows without area stay zspval."""
    nx, ny, nk, nb = 37, 6, 2, 2
    e1, e2, zm, mv, zv, alpha = zonal_exact(nx, ny, nk, nb, 11, general)
    assert _row_parts(nx, ny, 1, 3) == (3, 8, 2)
    zv[1, 2, :] = np.nan                              # every cell
    zv[1, 3, [0, 3, 18, 36]] = np.nan                 # head, first vector, body and tail of a row
    zv[1, 4, ::2] = np.nan
    zv[1, 4, 1::4] = 0.0                              # NaN and exact zeros
    mv[1, 2, :] = 1.0
    zm[2, :, :] = 1.0
    check_zonal(e1, e2, zm, mv, [zv], alpha)
    mean, zmax, zmin = oracle.zonalmean_record(zm, mv, zv, oracle.zonal_dlsurf(e1, e2), ZSP, True)
    assert np.isnan(mean[:, 1, 2:5]).all()
    assert np.all(zmax[:, 1, 2] == np.float32(-1.e20)) and np.all(zmin[:, 1, 2] == np.float32(1.e20))
    fin = np.where(np.isnan(zv[1, 3]), -np.inf, zv[1, 3])
    wet = zm[3, :, 0] * mv[1, 3] != 0                 # dry cells contribute dtmp = 0 to the max
    assert zmax[0, 1, 3] == max(fin[wet].max(), 0.0 if (~wet).any() else -np.inf)


@pytest.mark.parametrize("general", [None, 0.5], ids=["bits", "half"])
@pytest.mark.parametrize("nx", [129, 1442, 4322])
def test_k4_random_against_fsum(nx, general):
    """Random data and metrics.  K4's longest chain: a lane adds its head / tail cell and 4 cells per vector trip,
    then 5 shuffle levels -> D = 4 ceil(nvec / 32) + 1 + 5."""
    ny, nk, nb = 3, 2, 3
    rng = np.random.default_rng(nx)
    e1 = (rng.random((ny, nx)) * 2e4 + 1e3).astype(np.float32)
    e2 = (rng.random((ny, nx)) * 2e4 + 1e3).astype(np.float32)
    mv = (rng.random((nk, ny, nx)) > 0.2).astype(np.float32)
    zm = (rng.random((ny, nx, nb)) > 0.4).astype(np.float32)
    if general is not None:
        zm[:, ::7, 1] = general
    zv = (rng.standard_normal((nk, ny, nx)) * 3 + 1).astype(np.float32)
    alpha = (rng.random(ny) + 0.5).astype(np.float32)
    D = 4 * math.ceil((nx // 4) / 32) + 1 + 5
    dl = (np.float64(1.0) * e1.astype(np.float64)) * e2.astype(np.float64)
    shape = lib.cdfzonal_setup(e1, e2, zm, mv)
    try:
        gs = lib.cdfzonal_sum(zv, shape, alpha)
        gm = lib.cdfzonal_mean(zv, shape, ZSP, False)[0]
    finally:
        lib.cdfzonal_teardown()
    for b in range(nb):
        for k in range(nk):
            m8 = zm[:, :, b].astype(np.float64)
            p = ((zm[:, :, b] * mv[k]).astype(np.float32) * zv[k]).astype(np.float32).astype(np.float64)
            ts = dl * p                                                     # cdfzonalsum terms
            tm = dl * (((1.0 * m8) * mv[k].astype(np.float64)) * zv[k].astype(np.float64))   # cdfzonalmean terms
            ta = (dl * m8) * mv[k].astype(np.float64)                       # area terms
            for j in range(ny):
                a = float(alpha[j])
                s, es = math.fsum(ts[j]) / a, 2 * gamma(D) * np.abs(ts[j]).sum() / a
                assert abs(gs[b, k, j] - s) <= es + 4 * U * abs(s), (b, k, j)
                area, ea = math.fsum(ta[j]), 2 * gamma(D) * np.abs(ta[j]).sum()
                if area == 0.0:
                    assert gm[b, k, j] == ZSP
                    continue
                mean, em = math.fsum(tm[j]) / area, 2 * gamma(D) * np.abs(tm[j]).sum()
                tol = (em + abs(mean) * ea) / (abs(area) - ea) + 4 * U * abs(mean)
                assert abs(gm[b, k, j] - mean) <= tol, (b, k, j)


# ---- K5: cdfmhst ---------------------------------------------------------------------------------------------------------
def mhst_exact(nx, ny, nz, seed):
    """-> e1v, e3v, vmask1, (atl, pac, ind), zvt, zvs.  Heat terms (zvt*e1v*e3v)*1000*4000 stay below 2^31 in multiples of
    4, so every partial sum of a row (<= 8 levels, <= 8192 columns) is exact in fp64."""
    rng = np.random.default_rng(seed)
    e1v, e3v = pow2(rng, (ny, nx)), pow2(rng, (nz, ny, nx))
    masks = [(rng.random((ny, nx)) > p).astype(np.float32) for p in (0.2, 0.6, 0.5, 0.7)]
    zvt = exact_field((nz, ny, nx), nbits=7)
    zvs = exact_field((nz, ny, nx), nbits=7, offset=12345)
    return e1v, e3v, masks[0], masks[1:], zvt, zvs


def check_mhst(e1v, e3v, v1, basins, zvt, zvs, zdim, with_basins):
    kw = dict(zip(("atl", "pac", "ind"), basins)) if with_basins else {}
    ref = oracle.mhst_record(e1v, e3v, v1, zvt, zvs, zdim=zdim, **kw)
    dims = lib.cdfmhst_setup(e1v, e3v, v1, **kw)
    try:
        got = lib.cdfmhst_record(zvt, zvs, dims, zdim)
    finally:
        lib.cdfmhst_teardown()
    assert same_bits(got[0], ref[0]), "heat"
    assert same_bits(got[1], ref[1]), "salt"
    return got


@pytest.mark.parametrize("basins", [True, False], ids=["basins", "global"])
@pytest.mark.parametrize("zdim", [False, True], ids=["last", "zdim"])
@pytest.mark.parametrize("nx", [1, 2, 3, 5, 255, 256, 257, 1442, 2048, 2049, 4096, 4097, 4322, 8192])
def test_k5_widths(nx, zdim, basins):
    """The column ownership i = tid + c * nthreads over the 256 / 512 / 1024-thread launches (up to 8 columns a thread,
    nx <= 8192), and with odd nx the cp.async head and tail take every misalignment as the levels go by."""
    e1v, e3v, v1, b3, zvt, zvs = mhst_exact(nx, 3, 4, nx)
    heat, salt = check_mhst(e1v, e3v, v1, b3, zvt, zvs, zdim, basins)
    if nx <= 2:   # the global sum runs over i = 2..nx-1: empty
        assert np.all(heat[:, 0] == 0.0) and np.all(salt[:, 0] == 0.0)
        assert not np.signbit(heat[:, 0]).any()
    else:
        assert np.count_nonzero(heat[:, 0]) > 0


def test_k5_rejects_more_than_8192_columns():
    e1v, e3v, v1, b3, zvt, zvs = mhst_exact(8193, 1, 2, 1)
    with pytest.raises(lib.CdfGpuError) as ei:
        lib.cdfmhst_setup(e1v, e3v, v1)
    assert ei.value.code == ERR_ARG
    dims = lib.cdfmhst_setup(e1v[:, :8192], e3v[:, :, :8192], v1[:, :8192])   # the limit itself is accepted
    lib.cdfmhst_teardown()
    assert dims == (2, 1)


@pytest.mark.parametrize("zdim", [False, True], ids=["last", "zdim"])
@pytest.mark.parametrize("nx", [5, 257])
def test_k5_blocks_loop_over_rows(nx, zdim):
    """ny = 2100 rows: more than the grid (SMs x resident blocks), so a block integrates several rows j in turn."""
    e1v, e3v, v1, b3, zvt, zvs = mhst_exact(nx, 2100, 3, 2100 + nx)
    check_mhst(e1v, e3v, v1, b3, zvt, zvs, zdim, True)


@pytest.mark.parametrize("zdim", [False, True], ids=["last", "zdim"])
@pytest.mark.parametrize("nx", [1442, 4322, 8192])
def test_k5_random_against_fsum(nx, zdim):
    """Random data.  The per-column vertical integral is the oracle's own chain (bit for bit); the zonal stage adds up to
    8 columns per thread, 5 shuffle levels and up to 32 warp partials in sequence: D <= 8 + 5 + 32."""
    ny, nz = 3, 5
    rng = np.random.default_rng(nx + zdim)
    f4, f8 = np.float32, np.float64
    e1v = (rng.random((ny, nx)) * 5e4 + 1e3).astype(f4)
    e3v = (rng.random((nz, ny, nx)) * 200 + 1).astype(f4)
    masks = [(rng.random((ny, nx)) > p).astype(f4) for p in (0.2, 0.6, 0.5, 0.7)]
    zvt = (rng.standard_normal((nz, ny, nx)) * 5 + 8).astype(f4)
    zvs = (rng.standard_normal((nz, ny, nx)) * 0.5 + 35).astype(f4)
    dims = lib.cdfmhst_setup(e1v, e3v, masks[0], *masks[1:])
    try:
        heat, salt = lib.cdfmhst_record(zvt, zvs, dims, zdim)
    finally:
        lib.cdfmhst_teardown()
    D = 8 + 5 + 32
    dtrph, dtrps = np.zeros((ny, nx), f8), np.zeros((ny, nx), f8)
    for k in range(nz):
        dtrph = dtrph + (((zvt[k] * e1v).astype(f4) * e3v[k]).astype(f4).astype(f8) * f8(1000.0)) * f8(4000.0)
        dtrps = dtrps + ((zvs[k] * e1v).astype(f4) * e3v[k]).astype(f4).astype(f8)
        if not (zdim or k == nz - 1):
            continue
        lev = k if zdim else 0
        for m, mk in enumerate(masks):
            i0, i1 = (1, nx - 1) if m == 0 else (0, nx)
            for got, acc in ((heat, dtrph), (salt, dtrps)):
                for j in range(ny):
                    t = acc[j, i0:i1] * mk[j, i0:i1].astype(f8)
                    ref = math.fsum(t)
                    assert abs(got[lev, m, j] - ref) <= 2 * gamma(D) * np.abs(t).sum(), (lev, m, j)


# ---- K5v: cdfmhst -v/-t[-s] ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("zdim", [False, True], ids=["last", "zdim"])
@pytest.mark.parametrize("shape", [(5, 1, 3), (1, 4, 3), (1, 1, 2), (37, 5, 4), (257, 3, 3)],
                         ids=["ny1", "nx1", "one-column", "odd", "257"])
def test_k5v_vpoint_edges(shape, zdim):
    """K5v's V-point products against the host loop (through the same K5: bit for bit), then against the oracle on
    the host products (exact data: bit for bit).  ny = 1: every row is the last one, written as 0."""
    nx, ny, nz = shape
    e1v, e3v, v1, b3, _, _ = mhst_exact(nx, ny, nz, nx * ny * nz)
    zv = exact_field((nz, ny, nx), nbits=5)
    zt = (exact_field((nz, ny, nx), nbits=6, offset=7) + np.float32(10.0)).astype(np.float32)
    zs = (exact_field((nz, ny, nx), nbits=6, offset=3) + np.float32(35.0)).astype(np.float32)
    kw = dict(zip(("atl", "pac", "ind"), b3))
    hvt, hvs = vpoint(zv, zt, zs)
    dims = lib.cdfmhst_setup(e1v, e3v, v1, **kw)
    try:
        got = lib.cdfmhst_record_vts(zv, zt, zs, dims, zdim)
        host = lib.cdfmhst_record(hvt, hvs, dims, zdim)
    finally:
        lib.cdfmhst_teardown()
    ref = oracle.mhst_record(e1v, e3v, v1, hvt, hvs, zdim=zdim, **kw)
    for g, h, r in zip(got, host, ref):
        assert same_bits(g, h) and same_bits(g, r)
    if ny == 1:
        assert np.all(got[0] == 0.0) and np.all(got[1] == 0.0)
    else:
        assert np.count_nonzero(got[0][:, 1:]) > 0


# ---- K6: cdftransig_xy3d -----------------------------------------------------------------------------------------------------
def transig_frames(nx, ny, nz, nframes, seed, anomalies=True):
    """-> e2u, e1v, e3u, e3v, frames [(zu, zv, zt, zs)].  A quarter of the velocities are 0 (the frames' masks); frame 1
    carries NaN and +-Inf in T and in S, T/S whose density falls below the table and above its top, and a NaN u and v."""
    rng = np.random.default_rng(seed)
    nzm1 = nz - 1
    f4 = np.float32
    e2u = (rng.random((ny, nx)) * 5e3 + 5e3).astype(f4)
    e1v = (rng.random((ny, nx)) * 5e3 + 5e3).astype(f4)
    e3u = (rng.random((nzm1, ny, nx)) * 100 + 5).astype(f4)
    e3v = (rng.random((nzm1, ny, nx)) * 100 + 5).astype(f4)
    frames = []
    for n in range(nframes):
        zu = (0.1 * rng.standard_normal((nzm1, ny, nx)) * (rng.random((nzm1, ny, nx)) > 0.25)).astype(f4)
        zv = (0.1 * rng.standard_normal((nzm1, ny, nx)) * (rng.random((nzm1, ny, nx)) > 0.25)).astype(f4)
        zt = (rng.random((nzm1, ny, nx)) * 25).astype(f4)
        zs = (34 + 2 * rng.random((nzm1, ny, nx))).astype(f4)
        if anomalies and n == 1:
            cells = rng.choice(nzm1 * ny * nx, size=min(12, nzm1 * ny * nx), replace=False)
            edits = [(zu, np.nan), (zv, np.nan), (zu, np.inf), (zv, -np.inf),
                     (zt, np.nan), (zs, np.inf), (zt, -np.inf), (zs, np.nan), (zt, np.inf), (zs, -np.inf),
                     ((zt, zs), (35.0, 2.0)),     # far below ds1min
                     ((zt, zs), (-2.0, 60.0))]    # above the top of every table
            for c, (arr, val) in zip(cells, edits):
                if isinstance(arr, tuple):
                    arr[0].flat[c], arr[1].flat[c] = val
                else:
                    arr.flat[c] = val
        frames.append((zu, zv, zt, zs))
    return e2u, e1v, e3u, e3v, frames


K6_SHAPES = [synth.GRIDS[g] for g in ("TINY", "ODD", "SMALL", "ORCA2")] + [
    (1, 4, 3), (2, 4, 3), (3, 4, 3), (9, 1, 3), (11, 5, 2), (1442, 6, 12)]
K6_IDS = ["TINY", "ODD", "SMALL", "ORCA2", "nx1", "nx2", "nx3", "ny1", "nz2", "orca025-band"]
K6_CFGS = [(0.0, CODES[0], False, False), (1000.0, CODES[1], True, False), (2000.0, CODES[3], True, True),
           (1000.0, CODES[4], False, False)]


@pytest.mark.parametrize("cfg", K6_CFGS, ids=["sigma0", "sigma1-perio", "sigma2-perio-teos10", "sigma1-zoom"])
@pytest.mark.parametrize("shape", K6_SHAPES, ids=K6_IDS)
def test_k6_bit_for_bit(shape, cfg):
    """Three frames, masks set by the first two; the accumulators equal the oracle's bit for bit (NaN where a
    non-finite transport was added).  Non-finite or out-of-range densities fall into the clamped first / last step."""
    pref, code, lperio, teos10 = cfg
    nx, ny, nz = shape
    nb, smin = code[0], code[1]
    e2u, e1v, e3u, e3v, frames = transig_frames(nx, ny, nz, 3, nx * 7 + ny + nz)
    _, _, itab, scm = lib.transig_bins(*code)
    ref_u, ref_v = np.zeros((nb, ny, nx)), np.zeros((nb, ny, nx))
    mu, mv = np.zeros(frames[0][0].shape, np.uint8), np.zeros(frames[0][0].shape, np.uint8)
    with np.errstate(all="ignore"):
        for n, (zu, zv, zt, zs) in enumerate(frames):
            oracle.transig_record(e2u, e1v, e3u, e3v, zu, zv, zt, zs, pref, smin, scm, itab, nb, ref_u, ref_v, mu, mv,
                                  n < 2, lperio, teos10)
    shp = lib.cdftransig_setup(e2u, e1v, e3u, e3v, nz, nb, pref, smin, scm, itab, lperio, teos10)
    try:
        for n, (zu, zv, zt, zs) in enumerate(frames):
            lib.cdftransig_record(zu, zv, zt, zs, set_masks=n < 2)
        du, dv = lib.cdftransig_fetch(shp)
    finally:
        lib.cdftransig_teardown()
    assert same_bits(du, ref_u), "dusigsig"
    assert same_bits(dv, ref_v), "dvsigsig"
    assert np.count_nonzero(ref_u) > 0 and np.isnan(ref_u).any() and np.isnan(ref_v).any()
