"""Latitude-band sharding of the sibling tools (cdfzonal, cdfmhst, cdftransig) under CDFGPU_SHARD=lat: every record split
over N devices gives, bit for bit, what one device gives -- on uneven bands, one-row bands, fewer rows than devices, the
halo row of the V-point kernels, every declared input storage, the record pipelines and the command-line twins -- while
each device holds only its band of the resident fields, slots and accumulators."""
import os
import subprocess

import numpy as np
import pytest

from cdftools_b200 import build, ncfiles, synth
from cdftools_b200.shard import band_plan
from test_gpu_packed import decoded, quantize
from test_gpu_sibling_inputs import MHST_OUTS, TRANSIG_KINDS, declare, handed, reset_siblings
from test_gpu_sibling_pipeline import TAGS, mhst_files, pipeline, same, transig_files, zonal_files

pytestmark = pytest.mark.gpu
ERR_STATE = 3
F4 = np.float32


@pytest.fixture
def lib(gpu_lib):
    reset_siblings(gpu_lib)
    yield gpu_lib
    reset_siblings(gpu_lib)
    gpu_lib.finalize()          # back to the session's context: one device, three slots
    gpu_lib.init(0, 3)


def need(lib, n):
    if lib.device_count() < n:
        pytest.skip(f"needs {n} GPUs")


def one_device(lib, nslots=3):
    lib.finalize()
    lib.init(0, nslots)


def bands(lib, n, nslots=3):
    lib.finalize()
    lib.init_multi(n, "lat", nslots)
    assert lib.num_devices() == n and lib.nslots() == nslots


NDEV = [2, 3]


# ---- inputs: seeded, any shape ----------------------------------------------------------------------------------------------
class Case:
    """Resident fields and records of the three tools on an (nx, ny, nz) grid; `hot` rows get NaN / Inf and extreme T / S."""

    def __init__(self, nx, ny, nz, seed=7, hot=(), nrec=3):
        rng = np.random.default_rng(seed)
        self.nx, self.ny, self.nz = nx, ny, nz
        u = lambda *s: rng.random(s, dtype=np.float64).astype(F4)
        self.e1, self.e2 = u(ny, nx) * 5e3 + 5e3, u(ny, nx) * 5e3 + 5e3
        self.zmask = (rng.random((ny, nx, 5)) > 0.3).astype(F4)
        self.zmask[::3, ::2, 1] = 0.5                      # some non-binary basin masks (the general K4 path) on some rows
        self.mvar = (rng.random((nz - 1, ny, nx)) > 0.2).astype(F4)
        self.alpha = (0.5 + np.arange(ny) / max(ny, 1)).astype(F4)
        self.e3 = u(nz, ny, nx) * 100 + 5
        self.vmask1, self.atl, self.pac, self.ind = ((rng.random((ny, nx)) > p).astype(F4) for p in (0.2, 0.5, 0.6, 0.7))
        self.recs = []
        for r in range(nrec):
            v = (0.1 * rng.standard_normal((nz, ny, nx)) * (rng.random((nz, ny, nx)) > 0.25)).astype(F4)
            uu = (0.1 * rng.standard_normal((nz, ny, nx)) * (rng.random((nz, ny, nx)) > 0.25)).astype(F4)
            t = (rng.random((nz, ny, nx)) * 28 - 1).astype(F4)
            s = (rng.random((nz, ny, nx)) * 4 + 33).astype(F4)
            for j in hot:                                  # the first row of a band: what the band above reads through its halo
                for k in range(nz):
                    i = (k + r) % nx
                    t[k, j, i], s[k, j, (i + 1) % nx] = (np.nan, np.inf, -np.inf, 60.0, -5.0)[k % 5], (np.nan, 0.0, 50.0, -np.inf)[k % 4]
                    t[k, j, (i + 2) % nx] = 1e30
                    v[k, j, (i + 3) % nx] = np.inf
            self.recs.append((uu, v, t, s))

    def zonal(self, lib):
        shape = lib.cdfzonal_setup(self.e1, self.e2, self.zmask, self.mvar)
        out = []
        for _, v, _, _ in self.recs:
            z = v[:-1]
            out += [lib.cdfzonal_sum(z, shape), lib.cdfzonal_sum(z, shape, self.alpha), lib.cdfzonal_mean(z, shape, 99999.0, False),
                    lib.cdfzonal_mean(z, shape, 99999.0, True)]
        lib.cdfzonal_teardown()
        return out

    def mhst(self, lib, basins=True):
        b = (self.atl, self.pac, self.ind) if basins else (None, None, None)
        dims = lib.cdfmhst_setup(self.e1, self.e3, self.vmask1, *b)
        out = []
        for _, v, t, s in self.recs:
            for zdim in (False, True):
                with np.errstate(all="ignore"):
                    out.append(lib.cdfmhst_record(v * t, v * s, dims, zdim))
                out.append(lib.cdfmhst_record_vts(v, t, s, dims, zdim))
        lib.cdfmhst_teardown()
        return out

    def transig_setup(self, lib, vvl, lperio, code="1000"):
        pref, nb, smin, scal, zoom, smn = lib.TRANSIG_CODES[code]
        _, _, itab, step = lib.transig_bins(nb, smin, scal, zoom, smn)
        e3 = (None, None) if vvl else (self.e3[:-1], (self.e3[:-1] * F4(1.01)).astype(F4))
        return lib.cdftransig_setup(self.e2, self.e1, *e3, self.nz, nb, pref, smin, step, itab, lperio=lperio)

    def transig(self, lib, vvl, lperio):
        shape = self.transig_setup(lib, vvl, lperio)
        for r, (uu, v, t, s) in enumerate(self.recs):
            e3 = dict(e3u_vvl=self.e3[:-1] * F4(1 + r / 8), e3v_vvl=self.e3[:-1]) if vvl else {}
            lib.cdftransig_record(uu[:-1], v[:-1], t[:-1], s[:-1], set_masks=r < 2, **e3)
        out = lib.cdftransig_fetch(shape)
        lib.cdftransig_teardown()
        return out

    def all(self, lib):
        return (self.zonal(lib), self.mhst(lib), self.mhst(lib, basins=False),
                [self.transig(lib, vvl, lperio) for vvl in (False, True) for lperio in (False, True)])


def shapes(n):
    nx, ny, nz = synth.GRIDS["ODD"]
    return {"SMALL": synth.GRIDS["SMALL"], "ODD": (nx, ny, nz), "ny=N": (nx, n, nz), "ny=N+1": (nx, n + 1, nz),
            "ny<N": (nx, n - 1, nz), "nx=3": (3, 2 * n + 1, nz)}


# ---- 1. the ABI, bit for bit against one device ------------------------------------------------------------------------------
@pytest.mark.parametrize("grid", ["SMALL", "ODD", "ny=N", "ny=N+1", "ny<N", "nx=3"])
@pytest.mark.parametrize("n", NDEV)
def test_bands_equal_one_device(lib, n, grid):
    need(lib, n)
    c = Case(*shapes(n)[grid])
    one_device(lib)
    ref = c.all(lib)
    assert np.abs(ref[0][0]).max() > 0 and np.abs(ref[3][0][0]).max() > 0
    bands(lib, n)
    got = c.all(lib)
    for tool, a, b in zip(("zonal", "mhst", "mhst without basins", "transig"), got, ref):
        for r, (x, y) in enumerate(zip(a, b)):
            assert same(x, y), (tool, r)


# ---- 2. the halo row: non-finite and extreme T / S in the first row of every band but the first ------------------------------
@pytest.mark.parametrize("n", NDEV)
def test_halo_rows_carry_nonfinite_and_extreme_values(lib, n):
    need(lib, n)
    nx, ny, nz = 37, 4 * n + 1, 6
    hot = [j0 for j0, _ in band_plan(ny, n)[1:]]
    c = Case(nx, ny, nz, seed=11, hot=hot)
    one_device(lib)
    ref = c.mhst(lib), [c.transig(lib, vvl, lperio) for vvl in (False, True) for lperio in (False, True)]
    assert any(np.isnan(h[..., hot[0] - 1]).any() for h, _ in ref[0][1::2])   # the row above a band reads the NaN of the next
    bands(lib, n)
    got = c.mhst(lib), [c.transig(lib, vvl, lperio) for vvl in (False, True) for lperio in (False, True)]
    for a, b in zip(got, ref):
        for r, (x, y) in enumerate(zip(a, b)):
            assert same(x, y), r


# ---- 3. declared input storage across the band offsets --------------------------------------------------------------------
@pytest.mark.parametrize("n", NDEV)
def test_declared_inputs_across_band_offsets(lib, n):
    need(lib, n)
    m = synth.make_mesh("ODD")
    land = m.vmask == 0
    v = quantize(synth.make_v_record(m, 0), "v", land)
    t, s = synth.make_ts_record(m, 0)
    t, s = quantize(t, "t", m.tmask == 0), quantize(s, "s", m.tmask == 0)
    e3 = quantize((m.e3v_0 * F4(1.01)).astype(F4), "e3", np.zeros(land.shape, bool))
    e3[e3 == 32767] = 100
    c = Case(m.nx, m.ny, m.nz)

    def run(rep):
        out = []
        declare(lib, lib.CALL_ZONAL, 0, rep, "v")
        shape = lib.cdfzonal_setup(c.e1, c.e2, c.zmask, c.mvar)
        out.append(lib.cdfzonal_sum(handed(v[:-1], "v", rep), shape, c.alpha))
        lib.cdfzonal_teardown()
        dims = lib.cdfmhst_setup(c.e1, c.e3, c.vmask1, c.atl, c.pac, c.ind)
        for f in range(2):
            declare(lib, lib.CALL_MHST, f, rep, "t")
        out.append(lib.cdfmhst_record(handed(t, "t", rep), handed(s, "t", rep), dims, True))
        for f, kind in enumerate(("v", "t", "s")):
            declare(lib, lib.CALL_MHST_VTS, f, rep, kind)
        out.append(lib.cdfmhst_record_vts(handed(v, "v", rep), handed(t, "t", rep), handed(s, "s", rep), dims, True))
        lib.cdfmhst_teardown()
        for a in range(6):
            declare(lib, lib.CALL_TRANSIG, a, rep, TRANSIG_KINDS[a])
        shape = c.transig_setup(lib, True, False)
        fr = [v[:-1], v[::-1][:-1].copy(), t[:-1], s[:-1], e3[:-1], e3[1:].copy()]
        arg = [handed(np.ascontiguousarray(x), TRANSIG_KINDS[a], rep) for a, x in enumerate(fr)]
        lib.cdftransig_record(*arg[:4], set_masks=True, e3u_vvl=arg[4], e3v_vvl=arg[5])
        out.append(lib.cdftransig_fetch(shape))
        lib.cdftransig_teardown()
        reset_siblings(lib)
        return out

    one_device(lib)
    ref = run("f32")
    bands(lib, n)
    for rep in ("f32", "f32be", "i16", "i16be"):
        got = run(rep)
        for r, (x, y) in enumerate(zip(got, ref)):
            assert same(x, y), (rep, r)


# ---- 4. the record pipelines under lat ------------------------------------------------------------------------------------
@pytest.mark.parametrize("nslots", [1, 3])
@pytest.mark.parametrize("n", NDEV)
def test_pipelines_under_bands_equal_the_synchronous_loop(lib, n, nslots):
    need(lib, n)
    c = Case(*synth.GRIDS["SMALL"], seed=5)
    c.recs = c.recs * 3                                   # more records than slots
    nrec = 2 * nslots + 1
    one_device(lib)
    zref = c.zonal(lib)
    mref = c.mhst(lib)
    tref = [c.transig(lib, vvl, False) for vvl in (False, True)]
    bands(lib, n, nslots)
    shape = lib.cdfzonal_setup(c.e1, c.e2, c.zmask, c.mvar)
    recs = [x[1][:-1] for x in c.recs[:nrec]]
    got = pipeline(lib, nrec, lambda s, r: lib.cdfzonal_submit_sum(s, recs[r], c.alpha), lambda s: lib.cdfzonal_fetch(s, shape))
    assert all(same(got[r], zref[4 * r + 1]) for r in range(nrec))
    got = pipeline(lib, nrec, lambda s, r: lib.cdfzonal_submit_mean(s, recs[r], 99999.0, True), lambda s: lib.cdfzonal_fetch(s, shape))
    assert all(same(got[r], zref[4 * r + 3]) for r in range(nrec))
    assert lib.cdfzonal_kernel_ms() > 0
    lib.cdfzonal_teardown()
    dims = lib.cdfmhst_setup(c.e1, c.e3, c.vmask1, c.atl, c.pac, c.ind)
    got = pipeline(lib, nrec, lambda s, r: lib.cdfmhst_submit_vts(s, *c.recs[r][1:], True), lambda s: lib.cdfmhst_fetch(s, dims))
    assert all(same(got[r], mref[4 * r + 3]) for r in range(nrec))
    assert lib.cdfmhst_kernel_ms() > 0
    lib.cdfmhst_teardown()
    for vvl, ref in zip((False, True), tref):
        shape = c.transig_setup(lib, vvl, False)
        held = [None] * nslots
        for r, (uu, v, t, s) in enumerate(c.recs):
            slot = r % nslots
            if r >= nslots:
                lib.cdftransig_wait(slot)
                for a in held[slot]:
                    a[:] = np.nan                        # refilled once the wait returns
            e3 = [c.e3[:-1] * F4(1 + r / 8), c.e3[:-1]] if vvl else []
            held[slot] = [np.array(x) for x in (uu[:-1], v[:-1], t[:-1], s[:-1], *e3)]
            k = dict(e3u_vvl=held[slot][4], e3v_vvl=held[slot][5]) if vvl else {}
            lib.cdftransig_submit(slot, *held[slot][:4], set_masks=r < 2, **k)
        assert lib.cdftransig_kernel_ms() > 0
        got = lib.cdftransig_fetch(shape)
        lib.cdftransig_teardown()
        assert same(got, ref), vvl


# ---- 5. the work is really split ------------------------------------------------------------------------------------------
def test_each_device_holds_its_band_only(lib):
    need(lib, 2)
    import torch
    n = min(lib.device_count(), 4)
    c = Case(1442, 400, 31, seed=3, nrec=1)

    def used(run):
        """device memory each device gained while `run` set a tool up and went through slot 1 (run returns the teardown)"""
        for d in range(n):
            torch.cuda.mem_get_info(d)
        free0 = [torch.cuda.mem_get_info(d)[0] for d in range(n)]
        teardown = run()
        got = [free0[d] - torch.cuda.mem_get_info(d)[0] for d in range(n)]
        teardown()
        return got

    uu, v, t, s = (x[:-1] for x in c.recs[0])

    def transig():
        shape = c.transig_setup(lib, False, False, code="2000")   # 174 bins: 2 x 0.8 GB of accumulators
        lib.cdftransig_submit(1, uu, v, t, s, set_masks=True)
        lib.cdftransig_fetch(shape)
        return lib.cdftransig_teardown

    def zonal():
        shape = lib.cdfzonal_setup(c.e1, c.e2, c.zmask, c.mvar)
        lib.cdfzonal_submit_sum(1, v, c.alpha)
        lib.cdfzonal_fetch(1, shape)
        return lib.cdfzonal_teardown

    def mhst():
        dims = lib.cdfmhst_setup(c.e1, c.e3, c.vmask1, c.atl, c.pac, c.ind)
        lib.cdfmhst_submit_vts(1, *c.recs[0][1:])
        lib.cdfmhst_fetch(1, dims)
        return lib.cdfmhst_teardown

    rows = [j1 - j0 for j0, j1 in band_plan(c.ny, n)]
    for name, run, halo in (("transig", transig, 1), ("zonal", zonal, 0), ("mhst", mhst, 1)):
        one_device(lib)
        whole = used(run)[0]
        assert whole > (1e9 if name == "transig" else 2e8), (name, whole)
        bands(lib, n)
        got = used(run)
        for d in range(n):
            want = whole * (rows[d] + (halo if d < n - 1 else 0)) / c.ny
            assert abs(got[d] - want) < 0.05 * want + (32 << 20), (name, d, got, want)
        assert got[0] < 0.6 * whole, (name, got, whole)


# ---- 6. command-line twins ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tools():
    return build.build_host()


def test_cli_bands_write_the_same_files(lib, tools, tmp_path):
    need(lib, 2)
    m = synth.make_mesh("SMALL")
    from test_gpu_sibling_inputs import transig_frames
    frames = transig_frames(m, 6)
    runs = (("cdfzonalsum_gpu", ["-f", "in.nc", "-p", "V", "-b", "new_maskglo.nc"], ["zonalsum.nc"]),
            ("cdfzonalmean_gpu", ["-f", "in.nc", "-p", "V", "-b", "new_maskglo.nc", "-max"], ["zonalmean.nc"]),
            ("cdfmhst_gpu", ["-v", "gridV.nc", "-t", "gridT.nc", "-s", "gridS.nc", "-MST"], MHST_OUTS),
            ("cdftransig_xy3d_gpu", ["-c", "SYN-B200", "-l", *TAGS, "-S", "-o", "uv.nc"], ["uv.nc"]))
    for how in ("packed", "float"):
        for ndev in ("1", "2"):
            d = tmp_path / how / ndev
            ncfiles.write_mesh(m, d)
            zonal_files(m, d, 5, how)
            mhst_files(m, d, 4, how)
            transig_files(m, d, frames, how, TAGS)
            e = dict(os.environ, CDFGPU_DEVICES=ndev, CDFGPU_SHARD="lat")
            for tool, args, _ in runs:
                r = subprocess.run([str(tools[tool])] + args, capture_output=True, text=True, cwd=d, env=e, timeout=600)
                assert r.returncode == 0, r.stdout + r.stderr
        for _, _, outs in runs:
            for out in outs:
                assert (tmp_path / how / "1" / out).read_bytes() == (tmp_path / how / "2" / out).read_bytes(), (how, out)


# ---- 7. the *_device entry points still refuse several devices -------------------------------------------------------------
def test_device_entry_points_refuse_bands(lib):
    need(lib, 2)
    c = Case(37, 9, 5)
    bands(lib, 2)
    lib.cdfzonal_setup(c.e1, c.e2, c.zmask, c.mvar)
    lib.cdfmhst_setup(c.e1, c.e3, c.vmask1)
    c.transig_setup(lib, False, False)
    L = lib.load()
    calls = (lambda: L.cdfzonal_gpu_sum_device(None, None, None, None),
             lambda: L.cdfzonal_gpu_mean_device(None, 0.0, 0, None, None, None, None),
             lambda: L.cdfmhst_gpu_record_device(None, None, 0, None, None, None),
             lambda: L.cdfmhst_gpu_record_vts_device(None, None, None, 0, None, None, None),
             lambda: L.cdftransig_gpu_record_device(None, None, None, None, None, None, 0, None),
             lambda: L.cdftransig_gpu_fetch_device(None, None, None))
    for call in calls:
        assert call() == ERR_STATE
    lib.cdfzonal_teardown()
    lib.cdfmhst_teardown()
    lib.cdftransig_teardown()
