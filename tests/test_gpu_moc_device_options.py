"""cdfmoc -decomp, cdfmocsig -isodep and the cdfmaxmoc window search on device-resident records (cdfmoc_gpu_decomp_device,
cdfmocsig_gpu_compute_device_isodep, cdfmoc_gpu_maxmoc_windows / _device).

Each device call runs the kernels of its host-array twin, so the results are compared with that twin bit for bit: the four
-decomp slabs with decomp_submit / decomp_fetch, the -isodep depths with fetch_isodep (K2 with one chunk of levels per row,
whose histograms fold in a fixed order), every window of one maxmoc_device call with cdfmoc_gpu_maxmoc on the same slab.
The oracle checks the device results directly where a case is new.  Every record is seeded."""
import numpy as np
import pytest

import oracle
from cdftools_b200 import lib, synth
from test_gpu_moc_option_edges import (basins_from_five, bins_for, check_decomp, check_iso, decomp_ref, decomp_run,
                                       decomp_setup, iso_ref, mesh_case, mesh_record, random_case, same_result)
from util import assert_psi_close, case_inputs

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_STATE = 2, 3          # CDFGPU_ERR_ARG, CDFGPU_ERR_STATE
F4 = np.float32
KEYS = ("total", "sh", "bt", "ag")


@pytest.fixture(scope="module", autouse=True)
def _ctx(gpu_lib, oracle_mod):
    """The session-wide library context (conftest.gpu_lib), never finalised here: the test modules that follow use it."""
    yield
    lib.set_device_inputs_ready(False)


def torch_mod():
    import torch
    return torch


def to_dev(a):
    return torch_mod().from_numpy(np.ascontiguousarray(a)).cuda()


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def decomp_device(shape, rec, stream=None, producer=False):
    """decomp_device on device copies of rec -> dict of numpy slabs.  stream: None (the library's) or a torch stream.
    producer: the inputs are written by a torch kernel on `stream` right before the call."""
    torch = torch_mod()
    src = [to_dev(a) for a in rec]
    outs = {k: torch.full(shape, 7.0, dtype=torch.float64, device="cuda") for k in KEYS}
    torch.cuda.synchronize()
    if stream is None:
        lib.cdfmoc_decomp_device(*src, outs["total"], outs["sh"], outs["bt"], outs["ag"])
        lib.synchronize()
    else:
        with torch.cuda.stream(stream):
            if producer:
                dst = [torch.empty_like(a) for a in src]
                torch.cuda.synchronize()
                for d, a in zip(dst, src):
                    torch.mul(a, 1.0, out=d)       # a kernel on the caller stream writes the record
                src = dst
            lib.cdfmoc_decomp_device(*src, outs["total"], outs["sh"], outs["bt"], outs["ag"], stream=stream)
        stream.synchronize()
    return {k: v.cpu().numpy() for k, v in outs.items()}


def check_same(dev, host, what):
    for k in KEYS:
        assert same_bits(dev[k], host[k]), f"{what}: {k} differs from decomp_fetch"


def device_vs_host(c, rec, what, streams=(None, "torch")):
    shape = decomp_setup(c)
    host = decomp_run(shape, rec)
    for st in streams:
        dev = decomp_device(shape, rec, None if st is None else torch_mod().cuda.Stream())
        check_same(dev, host, f"{what} stream={st}")
    return host


# ---- 1. -decomp -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nb", range(1, 9))
def test_decomp_device_basin_counts(nb):
    m = synth.make_mesh("SMALL")
    c = mesh_case(m, basins_from_five(case_inputs(oracle, m, synth)[0], nb))
    rec = mesh_record(m, 60 + nb)
    host = device_vs_host(c, rec, f"nb={nb}", streams=(None, "torch") if nb in (1, 5, 8) else ("torch",))
    check_decomp(host, decomp_ref(c, rec), f"nb={nb}")


def test_decomp_device_nonbinary_masks():
    m = synth.make_mesh("SMALL")
    ib = case_inputs(oracle, m, synth)[0].copy()
    ib[:, :, 1] *= 3
    ib[::2, :, 4] *= -2
    c, rec = mesh_case(m, ib), mesh_record(m, 70)
    shape = decomp_setup(c)
    dev = decomp_device(shape, rec, torch_mod().cuda.Stream())
    check_same(dev, decomp_run(shape, rec), "non-binary masks")
    check_decomp(dev, decomp_ref(c, rec), "non-binary masks")


@pytest.mark.parametrize("shape", [(37, 9, 6), (1, 5, 4), (2, 6, 4), (9, 1, 4), (9, 2, 4), (37, 9, 2)],
                         ids=["37x9x6", "nx1", "nx2", "ny1", "ny2", "nz2"])
def test_decomp_device_wet_borders(shape):
    nx, ny, nz = shape
    c, rec = random_case(nx, ny, nz, 3, nx * 100 + ny * 10 + nz + 1)
    host = device_vs_host(c, rec, f"{shape}")
    check_decomp(host, decomp_ref(c, rec), f"{shape}")


def test_decomp_device_nonfinite_inputs():
    """NaN and +-Inf in V, T and S."""
    m = synth.make_mesh("SMALL")
    c = mesh_case(m)
    v, t, s = (a.copy() for a in mesh_record(m, 71))
    wet = np.argwhere(c.e3m[: m.nz - 1] * (c.ib[None, :, :, 0] != 0) > 0)
    v[tuple(wet[50])], v[tuple(wet[400])], v[tuple(wet[900])] = np.nan, np.inf, -np.inf
    t[tuple(wet[1500])], t[tuple(wet[1600])] = np.nan, np.inf
    s[tuple(wet[1700])], s[tuple(wet[1800])] = -np.inf, np.nan
    host = device_vs_host(c, (v, t, s), "non-finite")
    ref = decomp_ref(c, (v, t, s))
    check_decomp(host, ref, "non-finite")
    assert all(np.isnan(ref[k]).any() for k in KEYS)


@pytest.mark.parametrize("grid", [(1442, 24, 75), (4322, 8, 75)], ids=["orca025-width", "orca12-width"])
def test_decomp_device_production_widths(grid):
    m = synth.make_mesh(grid)
    c, rec = mesh_case(m, teos10=grid[0] == 4322), mesh_record(m, 72)
    shape = decomp_setup(c)
    dev = decomp_device(shape, rec, torch_mod().cuda.Stream())
    check_same(dev, decomp_run(shape, rec), f"{grid}")
    check_decomp(dev, decomp_ref(c, rec), f"{grid}")


def test_decomp_device_vvl_between_calls():
    """cdfmoc_set_e3v between device calls on a caller stream: the call after it reads the new e3m and area field."""
    m = synth.make_mesh("SMALL")
    c, rec = mesh_case(m), mesh_record(m, 73)
    e3b = (c.e3m * F4(1.0625)).astype(F4)
    e3b[: m.nz - 1][(c.e3m[: m.nz - 1] == 0) & (np.arange(m.nx)[None, None, :] % 5 == 0)] = F4(40.0)
    shape = decomp_setup(c)
    st = torch_mod().cuda.Stream()
    first = decomp_device(shape, rec, st)
    check_decomp(first, decomp_ref(c, rec), "before set_e3v")
    lib.cdfmoc_set_e3v(e3b)
    second = decomp_device(shape, rec, st)
    check_same(second, decomp_run(shape, rec, jt=1), "after set_e3v")
    check_decomp(second, decomp_ref(c, rec, e3b), "after set_e3v")


def test_decomp_device_inputs_from_a_kernel():
    """V, T and S written by a torch kernel on the caller stream right before the call (inputs not declared ready)."""
    m = synth.make_mesh("ODD")
    c, rec = mesh_case(m), mesh_record(m, 74, adversarial=True)
    shape = decomp_setup(c)
    host = decomp_run(shape, rec)
    for _ in range(3):
        check_same(decomp_device(shape, rec, torch_mod().cuda.Stream(), producer=True), host, "producer kernel")


def test_decomp_device_beside_the_slot_path():
    """Device calls and slot decompositions in turn share the plan's working fields: every result stays its own."""
    m = synth.make_mesh("ODD")
    c = mesh_case(m)
    recs = [mesh_record(m, 75 + r) for r in range(3)]
    shape = decomp_setup(c)
    hosts = [decomp_run(shape, recs[r], r % 2, r) for r in range(3)]
    torch = torch_mod()
    st = torch.cuda.Stream()
    srcs = [[to_dev(a) for a in r] for r in recs]
    outs = [{k: torch.empty(shape, dtype=torch.float64, device="cuda") for k in KEYS} for _ in recs]
    torch.cuda.synchronize()
    for n in range(3):
        lib.cdfmoc_decomp_submit(n % 2, n, *(np.ascontiguousarray(a) for a in recs[n]))
        lib.cdfmoc_decomp_device(*srcs[n], *(outs[n][k] for k in KEYS), stream=st)
        got = lib.cdfmoc_decomp_fetch(n % 2, shape)
        check_same(got, hosts[n], f"slot record {n}")
    st.synchronize()
    for n in range(3):
        check_same({k: v.cpu().numpy() for k, v in outs[n].items()}, hosts[n], f"device record {n}")


def test_decomp_device_launches_do_not_grow_with_depth():
    """decomp_device and decomp_submit each take the same number of launches at nz = 3 and nz = 76."""
    counts = {}
    for nz in (3, 76):
        c, rec = random_case(40, 12, nz, 3, nz)
        shape = decomp_setup(c)
        n0 = lib.launch_count()
        decomp_run(shape, rec)
        n1 = lib.launch_count()
        decomp_device(shape, rec, torch_mod().cuda.Stream())
        counts[nz] = (n1 - n0, lib.launch_count() - n1)
    assert counts[3] == counts[76], counts
    assert counts[3][1] == 11, counts       # K1 twice + nine -decomp kernels


def test_decomp_device_errors():
    torch = torch_mod()
    m = synth.make_mesh("ODD")
    c = mesh_case(m)
    shape = lib.cdfmoc_setup(c.e1v, c.e3m, c.ib)
    n3 = (m.nz - 1) * m.ny * m.nx
    src = [torch.zeros(n3, dtype=torch.float32, device="cuda") for _ in range(3)]
    outs = [torch.zeros(shape, dtype=torch.float64, device="cuda") for _ in KEYS]
    with pytest.raises(lib.CdfGpuError) as e:           # no decomp_setup
        lib.cdfmoc_decomp_device(*src, *outs)
    assert e.value.code == ERR_STATE
    lib.cdfmoc_decomp_setup(c.e1u, c.gphiv, c.gdept, c.um, c.tm)
    big = torch.zeros(n3 + 4, dtype=torch.float32, device="cuda")
    with pytest.raises(lib.CdfGpuError) as e:           # misaligned V
        lib.cdfmoc_decomp_device(big.data_ptr() + 4, src[1], src[2], *outs)
    assert e.value.code == ERR_ARG
    with pytest.raises(lib.CdfGpuError) as e:           # null output
        lib.cdfmoc_decomp_device(*src, outs[0], 0, outs[2], outs[3])
    assert e.value.code == ERR_ARG
    with pytest.raises(ValueError):                     # wrong element count, caught by the wrapper
        lib.cdfmoc_decomp_device(src[0][:-1], src[1], src[2], *outs)


# ---- 2. -isodep -------------------------------------------------------------------------------------------------------------
def isodep_both(e1v, e3v, ib, gdept, nz, v, t, s, cfg, eiv=None, e3r=None, stream="torch"):
    """The slot path (submit / fetch / fetch_isodep) and the device calls on the same record -> (slot, device, plain)
    where plain is cdfmocsig_compute_device's dmoc."""
    torch = torch_mod()
    pref, eos, smin, sstp, nbins = cfg
    shape = lib.cdfmocsig_setup(e1v, None if e3r is not None else e3v, ib, nz, nbins, smin, sstp, pref, eos)
    lib.cdfmocsig_set_isodep(gdept)
    moc, iso = np.empty(shape), np.empty(shape)
    lib.cdfmocsig_submit(0, 0, v, t, s, eiv, e3r)
    lib.cdfmocsig_fetch(0, moc)
    lib.cdfmocsig_fetch_isodep(0, iso)
    d = [to_dev(a) if a is not None else None for a in (v, t, s, eiv, e3r)]
    o = [torch.full(shape, 3.0, dtype=torch.float64, device="cuda") for _ in range(3)]
    torch.cuda.synchronize()
    st = torch.cuda.Stream() if stream == "torch" else None
    lib.cdfmocsig_compute_device_isodep(d[0], d[1], d[2], o[0], o[1], d_zveiv=d[3], d_e3v_vvl=d[4], stream=st)
    lib.cdfmocsig_compute_device(d[0], d[1], d[2], o[2], d_zveiv=d[3], d_e3v_vvl=d[4], stream=st)
    if st is not None:
        st.synchronize()
    lib.synchronize()
    return (moc, iso), (o[0].cpu().numpy(), o[1].cpu().numpy()), o[2].cpu().numpy()


def check_iso_bits(slot, dev, plain, what):
    assert same_bits(dev[1], slot[1]), f"{what}: depi differs from fetch_isodep"
    assert same_bits(dev[0], plain), f"{what}: dmoc differs from cdfmocsig_compute_device"
    assert same_bits(dev[0], slot[0]), f"{what}: dmoc differs from fetch"


@pytest.mark.parametrize("pref", [0.0, 2000.0])
@pytest.mark.parametrize("eos", [0, 1, 2], ids=["eos80", "teos10", "neutral"])
def test_isodep_device_eos_and_pref(eos, pref, monkeypatch):
    monkeypatch.setenv("CDFGPU_K2_CHUNKS", "1")
    m = synth.make_mesh("SMALL")
    ib = case_inputs(oracle, m, synth)[0]
    v, t, s = mesh_record(m, 80)
    cfg = (pref, eos, *bins_for(pref, eos))
    slot, dev, plain = isodep_both(m.e1v, m.e3v_0, ib, m.gdept_1d, m.nz, v, t, s, cfg, stream=None if eos == 1 else "torch")
    check_iso_bits(slot, dev, plain, f"{cfg}")
    check_iso(dev, iso_ref(m.e1v, m.e3v_0, ib, m.gdept_1d, v, t, s, cfg), f"{cfg}")


def test_isodep_device_eiv_and_vvl(monkeypatch):
    monkeypatch.setenv("CDFGPU_K2_CHUNKS", "1")
    m = synth.make_mesh("SMALL")
    ib = case_inputs(oracle, m, synth)[0]
    cfg = (2000.0, 0, 30.0, 0.05, 158)
    v, t, s = mesh_record(m, 81)
    eiv = (0.01 * synth.make_v_record(m, 82)[:-1]).astype(F4)
    slot, dev, plain = isodep_both(m.e1v, m.e3v_0, ib, m.gdept_1d, m.nz, v, t, s, cfg, eiv=eiv)
    check_iso_bits(slot, dev, plain, "-eiv")
    check_iso(dev, iso_ref(m.e1v, m.e3v_0, ib, m.gdept_1d, v, t, s, cfg, eiv=eiv), "-eiv")
    e3a = (m.e3v_0 * F4(1.03125)).astype(F4)
    slot, dev, plain = isodep_both(m.e1v, None, ib, m.gdept_1d, m.nz, v, t, s, cfg, e3r=np.ascontiguousarray(e3a[:-1]))
    check_iso_bits(slot, dev, plain, "device e3v_vvl")
    check_iso(dev, iso_ref(m.e1v, e3a, ib, m.gdept_1d, v, t, s, cfg), "device e3v_vvl")


def test_isodep_device_forced_cta_shapes(monkeypatch):
    """CDFGPU_K2_WARPS x CDFGPU_K2_CHUNKS: bit for bit with one chunk per row, against the oracle with several."""
    m = synth.make_mesh("SMALL")
    ib = case_inputs(oracle, m, synth)[0]
    v, t, s = mesh_record(m, 83)
    cfg = (0.0, 0, 23.0, 0.05, 104)
    ref = iso_ref(m.e1v, m.e3v_0, ib, m.gdept_1d, v, t, s, cfg)
    for warps in (1, 4, 16):
        for chunks in (1, 3):
            monkeypatch.setenv("CDFGPU_K2_WARPS", str(warps))
            monkeypatch.setenv("CDFGPU_K2_CHUNKS", str(chunks))
            slot, dev, plain = isodep_both(m.e1v, m.e3v_0, ib, m.gdept_1d, m.nz, v, t, s, cfg)
            if chunks == 1:
                check_iso_bits(slot, dev, plain, f"warps {warps}")
            check_iso(dev, ref, f"warps {warps} chunks {chunks}")


def test_isodep_device_errors():
    torch = torch_mod()
    m = synth.make_mesh("ODD")
    ib = case_inputs(oracle, m, synth)[0]
    shape = lib.cdfmocsig_setup(m.e1v, m.e3v_0, ib, m.nz, 52, 23.0, 0.1, 0.0, 0)
    n3 = (m.nz - 1) * m.ny * m.nx
    d = [torch.zeros(n3, dtype=torch.float32, device="cuda") for _ in range(3)]
    o = [torch.zeros(shape, dtype=torch.float64, device="cuda") for _ in range(2)]
    with pytest.raises(lib.CdfGpuError) as e:           # -isodep not enabled
        lib.cdfmocsig_compute_device_isodep(*d, *o)
    assert e.value.code == ERR_STATE
    lib.cdfmocsig_set_isodep(m.gdept_1d)
    with pytest.raises(lib.CdfGpuError) as e:
        lib.cdfmocsig_compute_device_isodep(*d, o[0], 0)
    assert e.value.code == ERR_ARG
    big = torch.zeros(o[1].numel() + 2, dtype=torch.float64, device="cuda")
    with pytest.raises(lib.CdfGpuError) as e:
        lib.cdfmocsig_compute_device_isodep(*d, o[0], big.data_ptr() + 8)
    assert e.value.code == ERR_ARG
    lib.cdfmocsig_set_isodep(None)
    with pytest.raises(lib.CdfGpuError) as e:           # switched off again
        lib.cdfmocsig_compute_device_isodep(*d, *o)
    assert e.value.code == ERR_STATE


# ---- 3. cdfmaxmoc -----------------------------------------------------------------------------------------------------------
def run_windows(d_psi, wins, stream=None):
    torch = torch_mod()
    lib.cdfmoc_maxmoc_windows(wins)
    ovt = torch.full((len(wins), 2), 5.0, dtype=torch.float32, device="cuda")
    loc = torch.full((len(wins), 4), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    lib.cdfmoc_maxmoc_device(d_psi, ovt, loc, stream=stream)
    if stream is not None:
        stream.synchronize()
    lib.synchronize()
    ovt, loc = ovt.cpu().numpy(), loc.cpu().numpy()
    return [(ovt[w, 0], ovt[w, 1], tuple(loc[w, :2]), tuple(loc[w, 2:])) for w in range(len(wins))]


def first_zero_sign(psi, basin, win, ext):
    """The sign bit the documented rule gives a zero extremum: that of the first cell in (j fastest, k) order holding it."""
    w = psi[win[2] - 1:win[3], win[0] - 1:win[1], basin].astype(F4).ravel()
    hit = w[(w == ext) & ~np.isnan(w)]
    return bool(np.signbit(hit[0]))


def check_windows(psi, got, wins, slot=None):
    for (basin, *win), g in zip(wins, got):
        ref = oracle.maxmoc(psi[:, :, basin].astype(F4), *win)
        assert same_result(g, ref), (basin, win, g, ref)
        for ext in g[:2]:
            if ext == 0.0:
                assert bool(np.signbit(ext)) == first_zero_sign(psi, basin, win, ext), (basin, win, g)
        if slot is not None:
            s = lib.cdfmoc_maxmoc(slot, basin, *win)
            assert same_bits(np.array(g[:2], F4), np.array(s[:2], F4)) and g[2:] == s[2:], (basin, win, g, s)


def orca2_windows(m, nb):
    wins = []
    for basin in range(nb):
        wins += [(basin, 1, m.ny, 1, m.nz), (basin, 40, 40, 12, 12), (basin, 70, 70, 1, m.nz), (basin, 1, 3, 1, m.nz),
                 (basin, 1, 1, 5, 9), (basin, 20, 120, 2, 20)]
    return wins


def test_maxmoc_device_on_compute_device_slab():
    """Windows over every basin -- one cell, one latitude, the whole slab, the closed southern rows (a +0 plateau) -- of a
    slab cdfmoc_gpu_compute_device wrote on a caller stream: equal to the slot search on the same record, and the oracle."""
    torch = torch_mod()
    m = synth.make_mesh("ORCA2")
    ib, e3m = case_inputs(oracle, m, synth)
    v = synth.make_v_record(m, 90)[:-1]
    shape = lib.cdfmoc_setup(m.e1v, e3m, ib)
    lib.cdfmoc_submit(1, 0, v)
    psi = lib.cdfmoc_fetch(1, np.empty(shape))
    d_v, d_psi = to_dev(v), torch.empty(shape, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    st = torch.cuda.Stream()
    lib.cdfmoc_compute_device(d_v, d_psi, st)
    wins = orca2_windows(m, shape[2])
    got = run_windows(d_psi, wins, stream=st)          # stream-ordered after the K1 launch
    assert same_bits(d_psi.cpu().numpy(), psi)
    check_windows(psi, got, wins, slot=1)


def test_maxmoc_device_on_batch_slab():
    torch = torch_mod()
    m = synth.make_mesh("ODD")
    ib, e3m = case_inputs(oracle, m, synth)
    shape = lib.cdfmoc_setup(m.e1v, e3m, ib)
    recs = [synth.make_v_record(m, 91 + r)[:-1] for r in range(3)]
    d_v = [to_dev(r) for r in recs]
    d_o = [torch.empty(shape, dtype=torch.float64, device="cuda") for _ in recs]
    torch.cuda.synchronize()
    st = torch.cuda.Stream()
    lib.cdfmoc_compute_device_batch(d_v, d_o, st)
    wins = [(b, j0, j1, k0, k1) for b in range(shape[2]) for (j0, j1, k0, k1) in
            ((1, m.ny, 1, m.nz), (2, 2, 1, 1), (3, m.ny - 1, 2, m.nz - 1), (m.ny, m.ny, m.nz, m.nz))]
    for r in range(3):
        got = run_windows(d_o[r], wins, stream=st)
        check_windows(d_o[r].cpu().numpy(), got, wins)


def synthetic_slab(ny, nz, nb, seed):
    """A slab with ties, +-0 plateaus, all-NaN and all +-Inf windows (values a K1 run can produce: NaN / Inf rows)."""
    rng = np.random.default_rng(seed)
    psi = np.round(rng.standard_normal((nz, ny, nb)) * 4).astype(np.float64)   # few distinct values: ties everywhere
    psi[:, 0:3] = 0.0
    psi[1:3, 1, :] = -0.0                  # a -0 / +0 plateau, -0 first in some windows
    psi[:, 5] = np.nan
    psi[:, 6] = np.inf
    psi[:, 7] = -np.inf
    psi[2:, 8] = np.nan
    psi[:2, 8] = -np.inf
    return psi


def test_maxmoc_device_edge_values():
    torch = torch_mod()
    m = synth.make_mesh("ODD")
    ib, e3m = case_inputs(oracle, m, synth)
    nz, ny, nb = lib.cdfmoc_setup(m.e1v, e3m, ib)
    assert ny >= 9
    psi = synthetic_slab(ny, nz, nb, 92)
    d_psi = to_dev(psi)
    wins = []
    for b in range(nb):
        wins += [(b, 1, 3, 1, nz), (b, 2, 3, 1, nz), (b, 2, 2, 2, 3), (b, 6, 6, 1, nz), (b, 7, 7, 1, nz), (b, 8, 8, 1, nz),
                 (b, 9, 9, 1, nz), (b, 6, 8, 1, nz), (b, 1, ny, 1, nz), (b, 4, 4, 1, 1), (b, 1, ny, nz, nz)]
    got = run_windows(d_psi, wins)
    check_windows(psi, got, wins)
    by = dict(zip(wins, got))
    g = by[(0, 6, 6, 1, nz)]
    assert np.isnan(g[0]) and np.isnan(g[1]) and g[2] == g[3] == (6, 1)
    g = by[(0, 7, 7, 1, nz)]
    assert g[0] == g[1] == np.inf and g[2] == g[3] == (7, 1)
    g = by[(0, 2, 3, 1, nz)]
    assert g[0] == 0.0 and g[1] == 0.0


def test_maxmoc_device_errors():
    torch = torch_mod()
    m = synth.make_mesh("ODD")
    ib, e3m = case_inputs(oracle, m, synth)
    nz, ny, nb = lib.cdfmoc_setup(m.e1v, e3m, ib)
    d_psi = torch.zeros((nz, ny, nb), dtype=torch.float64, device="cuda")
    ovt = torch.zeros((1, 2), dtype=torch.float32, device="cuda")
    loc = torch.zeros((1, 4), dtype=torch.int32, device="cuda")
    with pytest.raises(lib.CdfGpuError) as e:           # no windows yet
        lib.cdfmoc_maxmoc_device(d_psi, ovt, loc)
    assert e.value.code == ERR_STATE
    for w in ((0, 5, 4, 1, nz), (0, 1, ny, 3, 2), (0, 0, ny, 1, nz), (0, 1, ny + 1, 1, nz), (0, 1, ny, 1, nz + 1),
              (nb, 1, ny, 1, nz), (-1, 1, ny, 1, nz)):
        with pytest.raises(lib.CdfGpuError) as e:
            lib.cdfmoc_maxmoc_windows([(0, 1, ny, 1, nz), w])
        assert e.value.code == ERR_ARG, w
    lib.cdfmoc_maxmoc_windows([(0, 1, ny, 1, nz)])
    lib.cdfmoc_maxmoc_device(d_psi, ovt, loc)
    lib.synchronize()
    with pytest.raises(lib.CdfGpuError) as e:
        lib.cdfmoc_maxmoc_device(d_psi.data_ptr() + 8, ovt, loc)
    assert e.value.code == ERR_ARG
    lib.cdfmoc_setup(m.e1v, e3m, ib)                    # a new plan drops the windows
    with pytest.raises(lib.CdfGpuError) as e:
        lib.cdfmoc_maxmoc_device(d_psi, ovt, loc)
    assert e.value.code == ERR_STATE


# ---- 4. no copies, fixed launches -------------------------------------------------------------------------------------------
# The trace runs in a process of its own.  Traced in the pytest process, it was followed by a trace in
# test_gpu_sibling_device.py that did not show the host-to-device copy that test uses as its control; in separate processes
# a trace of these calls followed by further traces records such copies.  The module's traces must not depend on what
# earlier modules traced.
_TRACE = """
import json, sys
from pathlib import Path
sys.path[:0] = [sys.argv[1], str(Path(sys.argv[1]) / "tests")]
import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile
import oracle
from cdftools_b200 import lib, synth
from util import case_inputs
from test_gpu_moc_option_edges import decomp_setup, mesh_case, mesh_record
oracle.build()
lib.init(0, 3)
m = synth.make_mesh("SMALL")
c, rec = mesh_case(m), mesh_record(m, 95)
shape = decomp_setup(c)
ib = case_inputs(oracle, m, synth)[0]
sshape = lib.cdfmocsig_setup(m.e1v, m.e3v_0, ib, m.nz, 52, 23.0, 0.1, 0.0, 0)
lib.cdfmocsig_set_isodep(m.gdept_1d)
lib.cdfmoc_maxmoc_windows([(b, 1, m.ny, 1, m.nz) for b in range(shape[2])] * 6)
dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
src = [dev(a) for a in rec]
outs = [torch.empty(shape, dtype=torch.float64, device="cuda") for _ in range(4)]
so = [torch.empty(sshape, dtype=torch.float64, device="cuda") for _ in range(2)]
ovt = torch.empty((6 * shape[2], 2), dtype=torch.float32, device="cuda")
loc = torch.empty((6 * shape[2], 4), dtype=torch.int32, device="cuda")
st = torch.cuda.Stream()
calls = lambda: (lib.cdfmoc_decomp_device(*src, *outs, stream=st),
                 lib.cdfmocsig_compute_device_isodep(*src, *so, stream=st),
                 lib.cdfmoc_maxmoc_device(outs[0], ovt, loc, stream=st))
torch.cuda.synchronize()
calls()                                              # warm-up: module loads, EOS table, K2 plan
st.synchronize()
n0 = lib.launch_count()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    calls()
    st.synchronize()
launches = lib.launch_count() - n0
names = [e.name for e in prof.events()]
with profile(activities=[ProfilerActivity.CUDA]) as control:   # what a copy looks like in such a trace
    torch.ones(4).cuda()
    torch.cuda.synchronize()
print(json.dumps({"launches": launches, "names": names, "control": [e.name for e in control.events()]}))
lib.finalize()
"""


def test_device_calls_make_no_copies():
    """A torch.profiler trace of decomp_device, compute_device_isodep and maxmoc_device on a caller stream: their kernels,
    and no HtoD / DtoH copy."""
    import json
    import os
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    r = subprocess.run([sys.executable, "-c", _TRACE, str(root)], capture_output=True, text=True, env=dict(os.environ))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    got = json.loads(r.stdout.strip().splitlines()[-1])
    assert got["launches"] == 11 + 1 + 1
    for k in ("decomp_sigma_kernel", "decomp_geo_column_kernel", "moc_zonal_scan_kernel", "mocsig_eos_hist_scan_kernel",
              "moc_window_extrema_kernel"):
        assert any(k in n for n in got["names"]), f"{k} not in the trace"
    copies = [n for n in got["names"] if "HtoD" in n or "DtoH" in n]
    assert not copies, copies
    assert any("HtoD" in n for n in got["control"]), "the trace would not show a copy"
