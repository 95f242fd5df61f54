"""K1 (moc_zonal_scan_kernel, cdfmoc) and K2 (mocsig_eos_hist_scan_kernel, cdfmocsig) under every work plan they can
take, at the widths, depths and bin counts where their shape changes, against the C oracle.

Both kernels are persistent grids that hand out work by tickets; the plan follows the shape of the problem and the
documented knobs (INTEGRATION.md section 7), which setup reads.  What each plan must give:
  * K1: the same bits under every knob -- a row's sum is a fixed lane assignment plus a fixed shuffle tree, and the
    column scan is sequential -- and the oracle within util.assert_psi_close.
  * K2: the oracle within tolerance under every shape; at a fixed chunking the same bits whatever the warps, CTAs, PDL
    or bin tier (every tier feeds the same key into the same slot).
Bins of cells that sit on a bin edge (found by bisection over float32 salinities with the numpy oracle) reach tiers 2
and 3 of K2's bin function, and must equal the oracle bit for bit.  Every record is seeded."""
import numpy as np
import pytest
import torch

import oracle
import oracle.np_oracle as npo
from cdftools_b200 import lib, synth
from util import BUDGET, assert_psi_close, case_inputs, smem_bytes

pytestmark = pytest.mark.gpu

ERR_ARG = 2   # CDFGPU_ERR_ARG
F4 = np.float32
K1_KNOBS = ("CDFGPU_K1_CHUNK", "CDFGPU_K1_TAIL", "CDFGPU_K1_PDL", "CDFGPU_K1_SPARE_SMS")
K2_KNOBS = ("CDFGPU_K2_WARPS", "CDFGPU_K2_CTAS", "CDFGPU_K2_CHUNKS", "CDFGPU_K2_PDL", "CDFGPU_K2_TIER1", "CDFGPU_EXACT_EOS")


@pytest.fixture(scope="module", autouse=True)
def _ctx(gpu_lib, oracle_mod):
    """The session-wide library context (conftest.gpu_lib), never finalised here: the test modules that follow use it."""
    yield


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def set_knobs(monkeypatch, names, knobs):
    for k in names:
        monkeypatch.delenv(k, raising=False)
    for k, v in knobs.items():
        monkeypatch.setenv(k, str(v))


# ---- K1 -----------------------------------------------------------------------------------------------------------------
def mesh_k1(grid, nrec=4):
    m = synth.make_mesh(grid)
    ib, e3m = case_inputs(oracle, m, synth)
    recs = [np.ascontiguousarray(synth.make_v_record(m, 60 + r, adversarial=r % 2 == 1)[:-1]) for r in range(nrec)]
    return m.e1v, e3m, ib, recs


def k1_plans(nz):
    sms = sm_count()
    plans = [("default", {})]
    plans += [(f"chunk {c}", {"CDFGPU_K1_CHUNK": c}) for c in (1, 2, 3, 4, 5, nz - 1, nz + 6)]
    plans += [(f"chunk 3 tail {d}", {"CDFGPU_K1_CHUNK": 3, "CDFGPU_K1_TAIL": d}) for d in (2, 4, 16)]
    plans += [("chunk 1 tail 2 (tail off)", {"CDFGPU_K1_CHUNK": 1, "CDFGPU_K1_TAIL": 2})]
    plans += [(f"pdl {p}", {"CDFGPU_K1_PDL": p}) for p in (0, 1)]
    # SMs - 1 spare: 3 CTAs = 24 warps for 32 ticket shards, so some shards drain only by stealing
    plans += [(f"spare {s}", {"CDFGPU_K1_SPARE_SMS": s}) for s in (0, sms - 1)]
    plans += [("spare, pdl 0, chunk 5 tail 4", {"CDFGPU_K1_SPARE_SMS": sms - 1, "CDFGPU_K1_PDL": 0, "CDFGPU_K1_CHUNK": 5,
                                                "CDFGPU_K1_TAIL": 4})]
    return plans


def k1_plan_outputs(e1v, e3m, ib, recs):
    """Under the knobs now set: one launch per record (submit / fetch), 48 back-to-back launches on one torch stream (the
    three ticket sets rotate), and batched launches of 1, 2, 4 and 73 records with inputs-ready 0 and 1.
    -> {name: (nz, ny, nb) array} with record r % len(recs) behind every name."""
    nz, ny, nb = lib.cdfmoc_setup(e1v, e3m, ib)
    out = {}
    for r, v in enumerate(recs):
        o = np.empty((nz, ny, nb))
        lib.cdfmoc_submit(r % 3, r, v)
        lib.cdfmoc_fetch(r % 3, o)
        out[f"single {r}"] = o
    n = len(recs)
    d_recs = [torch.from_numpy(v).cuda() for v in recs]
    seq = torch.full((48, nz, ny, nb), float("nan"), dtype=torch.float64, device="cuda")
    batches = {(ready, nrec): torch.full((nrec, nz, ny, nb), float("nan"), dtype=torch.float64, device="cuda")
               for ready in (0, 1) for nrec in (1, 2, 4, 73)}
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    try:
        with torch.cuda.stream(st):
            for k in range(48):
                lib.cdfmoc_compute_device(d_recs[k % n], seq[k], st)
            for (ready, nrec), b in batches.items():
                lib.set_device_inputs_ready(ready)
                lib.cdfmoc_compute_device_batch([d_recs[r % n] for r in range(nrec)], [b[r] for r in range(nrec)], st)
        st.synchronize()
    finally:
        lib.set_device_inputs_ready(False)
    s = seq.cpu().numpy()
    for k in range(48):
        out[f"launch {k} of 48 (record {k % n})"] = s[k]
    for (ready, nrec), b in batches.items():
        bb = b.cpu().numpy()
        for r in range(nrec):
            out[f"batch of {nrec}, ready {ready}, record {r}"] = bb[r]
    return out


def record_of(name, n):
    r = int(name.rsplit(" ", 1)[1].rstrip(")"))
    return r % n


@pytest.mark.parametrize("grid", ["ORCA2", (1442, 24, 75), (4322, 8, 75)], ids=["orca2", "1442x24x75", "4322x8x75"])
def test_k1_plans_bit_identical(monkeypatch, grid):
    """Every chunking (1..5, nz-1, past nz), the guided tail, PDL on and off, spare SMs, each as single, back-to-back and
    batched launches: bit for bit the default plan's single launch, which matches the oracle."""
    e1v, e3m, ib, recs = mesh_k1(grid)
    nz = e3m.shape[0]
    set_knobs(monkeypatch, K1_KNOBS, {})
    base = k1_plan_outputs(e1v, e3m, ib, recs)
    ref = [base[f"single {r}"] for r in range(len(recs))]
    for r, v in enumerate(recs):
        assert_psi_close(ref[r], oracle.cdfmoc_record(e1v, e3m, ib, v), f"{grid} default plan, record {r}")
    for plan, knobs in k1_plans(nz):
        set_knobs(monkeypatch, K1_KNOBS, knobs)
        got = base if plan == "default" else k1_plan_outputs(e1v, e3m, ib, recs)
        for name, o in got.items():
            assert np.array_equal(o, ref[record_of(name, len(recs))], equal_nan=True), f"{grid} {plan}: {name} differs"


def k1_case(nx, ny, nz, nb, seed, general):
    """Random metrics with dry cells (zero area), basin masks set on all four edges, the last basin all zero and (nb >= 3)
    the one before it a single cell; general: one row of non-binary mask values.  V with +-0, subnormals and one row whose
    finite values overflow the fp32 product (row_general_store)."""
    rng = np.random.default_rng(seed)
    e1v = (rng.random((ny, nx)) * 4e4 + 5e3).astype(F4)
    wet = rng.random((nz, ny, nx)) > 0.2
    e3m = np.where(wet, rng.random((nz, ny, nx)) * 200 + 5, 0).astype(F4)
    ib = (rng.random((ny, nx, nb)) > 0.4).astype(np.int16)
    ib[0], ib[-1], ib[:, 0], ib[:, -1] = 1, 1, 1, 1
    if nb >= 2:
        ib[:, :, nb - 1] = 0
    if nb >= 3:
        ib[:, :, nb - 2] = 0
        ib[ny // 2, nx // 2, nb - 2] = 1
    if general:
        ib[ny // 2, :, 0] = rng.integers(-3, 4, nx)
    v = (0.1 * rng.standard_normal((nz - 1, ny, nx))).astype(F4)
    flat = v.reshape(-1)
    pick = rng.random(flat.size)
    flat[pick < 0.05] = F4(0.0)
    flat[(pick >= 0.05) & (pick < 0.1)] = F4(-0.0)
    flat[(pick >= 0.1) & (pick < 0.15)] = (rng.choice([-1, 1], flat.size) * 1e-40).astype(F4)[(pick >= 0.1) & (pick < 0.15)]
    k, j = (nz - 1) // 2, ny - 1 - ny // 3
    v[k, j] = F4(1e36)
    e3m[k, j, 0], ib[j, 0, 0] = F4(50.0), 1          # at least one covered, wet cell of that row overflows
    return e1v, e3m, ib, v


NX_CLASSES = {c: [nx for nx in (*range(1, 10), 129, 130, 131, 132, 1442, 4095, 4096, 4097, 4322) if nx % 4 == c] for c in range(4)}


def k1_shapes():
    """Every nb = 1..8 meets every nx mod 4 class (the 16-byte vectors straddle row ends differently), each class
    cycling through its widths (4095 -> 4096 is the chunk 4 -> 1 switch), with ny in {1, 3, 7} and nz in {2, 3, 76, 122}."""
    out = []
    for nb in range(1, 9):
        for c in range(4):
            nxs = NX_CLASSES[c]
            out.append((nxs[nb % len(nxs)], (1, 3, 7)[(nb + c) % 3], (2, 3, 76, 122)[(nb + 2 * c) % 4], nb))
    return out


@pytest.mark.parametrize("nx,ny,nz,nb", k1_shapes())
def test_k1_shapes(nx, ny, nz, nb):
    general = (nx + nb) % 2 == 1
    e1v, e3m, ib, v = k1_case(nx, ny, nz, nb, 1000 * nb + nx + ny + nz, general)
    shape = lib.cdfmoc_setup(e1v, e3m, ib)
    got = np.empty(shape)
    lib.cdfmoc_submit(0, 0, v)
    lib.cdfmoc_fetch(0, got)
    with np.errstate(all="ignore"):
        ref = oracle.cdfmoc_record(e1v, e3m, ib, v)
    assert np.isinf(ref).any() or np.isnan(ref).any()       # the overflowing row reached the result
    assert_psi_close(got, ref, f"{nx}x{ny}x{nz} nb={nb} general={general}")


@pytest.mark.parametrize("grid", ["ORCA025", "ORCA12-band"])
def test_k1_whole_records_batched(grid):
    """A whole ORCA025 L75 record and a 4322-wide ORCA12 band, two records per batched launch: every row against the
    oracle."""
    m = synth.make_mesh("ORCA025") if grid == "ORCA025" else synth.make_mesh("ORCA12", rows=(1338, 1721))
    ib, e3m = case_inputs(oracle, m, synth)
    recs = [np.ascontiguousarray(synth.make_v_record(m, 70 + r, adversarial=r == 1)[:-1]) for r in range(2)]
    nz, ny, nb = lib.cdfmoc_setup(m.e1v, e3m, ib)
    d_recs = [torch.from_numpy(v).cuda() for v in recs]
    outs = torch.full((2, nz, ny, nb), float("nan"), dtype=torch.float64, device="cuda")
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(st):
        lib.cdfmoc_compute_device_batch(d_recs, [outs[0], outs[1]], st)
    st.synchronize()
    o = outs.cpu().numpy()
    del d_recs, outs
    for r, v in enumerate(recs):
        assert_psi_close(o[r], oracle.cdfmoc_record(m.e1v, e3m, ib, v), f"{grid} record {r}")


def test_k1_shared_memory_limit():
    """8 basins at the deepest column that fits the device's shared memory per block (narrow grid, 1 CTA per SM) match
    the oracle; one level more is refused by setup with CDFGPU_ERR_ARG before any launch, and the next valid setup and
    record work (no error of the refusal is left behind for them)."""
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    per_level = 8 * 8 * 8                        # 8 warps x 8 basins x 8 B
    nz = optin // per_level + 1
    nx, ny, nb = 40, 3, 8
    e1v, e3m, ib, v = k1_case(nx, ny, nz, nb, 77, False)

    def run():
        shape = lib.cdfmoc_setup(e1v, e3m, ib)
        got = np.empty(shape)
        lib.cdfmoc_submit(0, 0, v)
        lib.cdfmoc_fetch(0, got)
        return got

    with np.errstate(all="ignore"):
        ref = oracle.cdfmoc_record(e1v, e3m, ib, v)
    assert_psi_close(run(), ref, f"nb=8 nz={nz}")
    over = k1_case(nx, ny, nz + 1, nb, 78, False)
    n0 = lib.launch_count()
    with pytest.raises(lib.CdfGpuError) as e:
        lib.cdfmoc_setup(*over[:3])
    assert e.value.code == ERR_ARG and "shared memory" in str(e.value) and str(optin) in str(e.value), str(e.value)
    assert lib.launch_count() == n0, "the refusal must come before any launch"
    assert_psi_close(run(), ref, f"nb=8 nz={nz} after the refusal")


# ---- K2 -----------------------------------------------------------------------------------------------------------------
def k2_run(e1v, e3v, ib, nz, cfg, recs, spv=0.0, spt=0.0, sps=0.0, j0=0, nyg=None):
    """One setup (which reads the K2 knobs), then the records in turn on slots 0 / 1 -> list of (ny, nbins, nb)."""
    pref, eos, smin, sstp, nbins = cfg
    shape = lib.cdfmocsig_setup(e1v, e3v, ib, nz, nbins, smin, sstp, pref, eos, spv, spt, sps, j_first_global=j0, ny_global=nyg)
    outs = []
    for n, (v, t, s) in enumerate(recs):
        out = np.empty(shape)
        lib.cdfmocsig_submit(n % 2, n, v, t, s)
        lib.cdfmocsig_fetch(n % 2, out)
        outs.append(out)
    return outs


def k2_ref(e1v, e3v, ib, rec, cfg, spv=0.0, spt=0.0, sps=0.0):
    pref, eos, smin, sstp, nbins = cfg
    with np.errstate(all="ignore"):
        return oracle.cdfmocsig_record(e1v, e3v, ib, *rec, spv, spt, sps, pref, eos, smin, sstp, nbins, want_bins=False)[0]


def mesh_k2(m, rec):
    t, s = synth.make_ts_record(m, rec)
    return synth.make_v_record(m, rec)[:-1], t[:-1], s[:-1]


SIG0 = (0.0, 0, 23.0, 0.05, 104)
SIG2 = (2000.0, 0, 30.0, 0.05, 158)
NTR = (0.0, 2, 25.0, 0.05, 80)


@pytest.mark.parametrize("cfg", [SIG0, SIG2, NTR], ids=["eos80-sigma0", "eos80-sigma2000", "neutral"])
def test_k2_forced_shapes(monkeypatch, cfg):
    """CDFGPU_K2_WARPS x CDFGPU_K2_CHUNKS, and CDFGPU_K2_CTAS / CDFGPU_K2_PDL: every shape matches the oracle and is
    reproducible run to run; with one chunk per row the bits do not depend on the warps, the CTAs or PDL."""
    m = synth.make_mesh("SMALL")
    ib = case_inputs(oracle, m, synth)[0]
    rec = mesh_k2(m, 80)
    ref = k2_ref(m.e1v, m.e3v_0, ib, rec, cfg)
    nzm1 = m.nz - 1
    shapes = [{"CDFGPU_K2_WARPS": w, "CDFGPU_K2_CHUNKS": c} for w in (1, 2, 4, 8, 16) for c in (1, 3, nzm1)]
    shapes += [{"CDFGPU_K2_WARPS": w, "CDFGPU_K2_CHUNKS": 1, "CDFGPU_K2_CTAS": n, "CDFGPU_K2_PDL": p}
               for w in (8, 16) for n in (1, 2) for p in (0, 1)]
    one_chunk = []
    for knobs in shapes:
        set_knobs(monkeypatch, K2_KNOBS, knobs)
        got = k2_run(m.e1v, m.e3v_0, ib, m.nz, cfg, [rec, rec])
        assert_psi_close(got[0], ref, f"{knobs}")
        assert np.array_equal(got[0], got[1], equal_nan=True), f"{knobs}: not reproducible"
        nkc = -(-nzm1 // knobs["CDFGPU_K2_CHUNKS"])
        info = lib.cdfmocsig_filter_info()
        assert info["chunks_per_row"] == -(-nzm1 // nkc) and info["levels_per_chunk"] == nkc, (knobs, info)
        if "CDFGPU_K2_CTAS" in knobs:
            assert info["resident_ctas"] <= knobs["CDFGPU_K2_CTAS"] * sm_count(), (knobs, info)
        if knobs["CDFGPU_K2_CHUNKS"] == 1:
            one_chunk.append((knobs, got[0]))
    differ = [k for k, o in one_chunk if not np.array_equal(o, one_chunk[0][1], equal_nan=True)]
    assert not differ, f"one chunk per row: {differ} differ from {one_chunk[0][0]}"


def random_k2(nx, ny, nz, ib, seed):
    rng = np.random.default_rng(seed)
    e1v = (rng.random((ny, nx)) * 4e4 + 5e3).astype(F4)
    e3v = (rng.random((nz, ny, nx)) * 200 + 5).astype(F4)
    v = (0.1 * rng.standard_normal((nz - 1, ny, nx))).astype(F4)
    t = (rng.random((nz - 1, ny, nx)) * 26 - 1).astype(F4)
    s = (rng.random((nz - 1, ny, nx)) * 3.5 + 33).astype(F4)
    return e1v, e3v, (v, t, s)


TUPLES = [[(p >> b) & 1 for b in range(5)] for p in range(1, 32)]


def k2_masks(nx, ny, ntup, seed):
    """(ny, nx, 5) masks: the counted cells (1 <= i <= nx-2) hold up to `ntup` distinct non-zero tuples, every 7th cell
    none; the excluded columns i = 0, nx-1 hold tuples too (they must not count)."""
    rng = np.random.default_rng(seed)
    ib = np.zeros((ny, nx, 5), np.int16)
    if ntup:
        cells = rng.permutation([(j, i) for j in range(ny) for i in range(1, nx - 1)])
        for n, (j, i) in enumerate(cells):
            if n % 7 != 6:
                ib[j, i] = TUPLES[n % ntup]
        ib[:, 0] = TUPLES[-1]
        ib[:, nx - 1] = TUPLES[3]
    return ib


def test_k2_automatic_shape_switch():
    """ny = 4 x SMs - 1 runs 16 warps x 1 CTA per SM, ny = 4 x SMs 8 warps x 2 CTAs (a narrow, tall grid: both shapes
    cheaply)."""
    sms = sm_count()
    resident = {}
    for ny in (4 * sms - 1, 4 * sms):
        ib = k2_masks(64, ny, 5, ny)
        e1v, e3v, rec = random_k2(64, ny, 10, ib, ny)
        got = k2_run(e1v, e3v, ib, 10, SIG0, [rec])[0]
        assert_psi_close(got, k2_ref(e1v, e3v, ib, rec, SIG0), f"ny={ny}")
        resident[ny] = lib.cdfmocsig_filter_info()["resident_ctas"]
    assert resident[4 * sms - 1] == sms and resident[4 * sms] == 2 * sms, resident


K2_NX = (1, 2, 3, 4, 5, 255, 256, 257, 258, 259, 513, 1442, 4322)
K2_NBINS = (1, 2, 7, 8, 9, 104, 158)


def k2_shapes():
    """Every width (K2 windows are 256 cells: nx = 0..3 mod 4 around 256 and 512) twice, with ny in {1, 2, 3} inside or
    outside a band, nz in {2, 3, 76}, the bin counts where the 8-bin lane table band runs past nbins, and 0, 1 or 31
    non-zero mask tuples."""
    out = []
    for n, nx in enumerate(K2_NX):
        for rep in range(2):
            q = 2 * n + rep
            ny = (1, 2, 3)[q % 3] if rep else (3, 3, 1, 2)[n % 4]     # outside a band only ny = 3 has a counted row
            out.append((nx, ny, (2, 3, 76)[(q // 3 + rep) % 3], K2_NBINS[q % 7], (0, 1, 31)[(n + 2 * rep) % 3], rep == 1))
    return out


@pytest.mark.parametrize("nx,ny,nz,nbins,ntup,band", k2_shapes())
def test_k2_shapes(nx, ny, nz, nbins, ntup, band):
    """A band (j_first_global > 0) counts all its rows; the oracle sees the band with one row of the whole domain on
    each side.  Without a band the first and last row are not counted (a single row is: jj = 2..npjglo-1 is empty, and the
    reference's loop then runs once); nx <= 2 has no counted column at all."""
    nyo = ny + 2 if band else ny
    ib = k2_masks(nx, nyo, ntup, nx + ny)
    e1v, e3v, rec = random_k2(nx, nyo, nz, ib, 7 * nx + nz)
    pref = 0.0 if nbins % 2 else 2000.0
    cfg = (pref, 0, 20.0 if pref == 0.0 else 30.0, 8.0 / nbins, nbins)
    ref = k2_ref(e1v, e3v, ib, rec, cfg)
    if band:
        b = slice(1, ny + 1)
        c2, c3 = (lambda a: np.ascontiguousarray(a[b])), (lambda a: np.ascontiguousarray(a[:, b]))
        got = k2_run(c2(e1v), c3(e3v), c2(ib), nz, cfg, [tuple(c3(a) for a in rec)], j0=5, nyg=5 + ny + 3)[0]
        ref = ref[b]
    else:
        got = k2_run(e1v, e3v, ib, nz, cfg, [rec])[0]
    assert_psi_close(got, ref, f"{nx}x{ny}x{nz} nbins={nbins} tuples={ntup} band={band}")
    if nx <= 2 or ntup == 0 or (ny == 2 and not band):
        assert np.all(got == 0.0)
    else:
        assert np.any(got != 0.0)


def test_k2_shared_memory_limit():
    """31 mask tuples and the largest bin count whose histogram fits one warp's CTA: the plan gives up warps (two would
    not fit) and matches the oracle; one bin more is refused by setup, and the next valid setup and record work."""
    nx, ny, nz = 64, 24, 6
    ib = k2_masks(nx, ny, 31, 9)
    fit = max(n for n in range(200, 2000) if smem_bytes(False, 1, n, 31, 5) <= BUDGET)
    assert smem_bytes(False, 2, fit, 31, 5) > BUDGET
    e1v, e3v, rec = random_k2(nx, ny, nz, ib, 10)
    cfg = (0.0, 0, 20.0, 8.0 / fit, fit)
    ref = k2_ref(e1v, e3v, ib, rec, cfg)
    assert_psi_close(k2_run(e1v, e3v, ib, nz, cfg, [rec])[0], ref, f"{fit} bins")
    with pytest.raises(lib.CdfGpuError) as e:
        lib.cdfmocsig_setup(e1v, e3v, ib, nz, fit + 1, 20.0, 8.0 / fit, 0.0, 0)
    assert e.value.code == ERR_ARG and "shared memory" in str(e.value)
    assert_psi_close(k2_run(e1v, e3v, ib, nz, cfg, [rec])[0], ref, f"{fit} bins after the refusal")


@pytest.mark.parametrize("grid", ["ORCA025", "ORCA12-band"])
def test_k2_whole_records(grid):
    """Every row against the oracle: ORCA025 L75 at sigma0 / 104 bins (8 warps x 2 CTAs per SM), and 383 rows of ORCA12
    at sigma2 / 158 bins (16 warps x 1 CTA per SM); both one chunk per row."""
    if grid == "ORCA025":
        m, cfg = synth.make_mesh("ORCA025"), SIG0
    else:
        m, cfg = synth.make_mesh("ORCA12", rows=(1338, 1721)), SIG2
    ib = case_inputs(oracle, m, synth)[0]
    rec = mesh_k2(m, 81)
    got = k2_run(m.e1v, m.e3v_0, ib, m.nz, cfg, [rec])[0]
    info = lib.cdfmocsig_filter_info()
    assert info["chunks_per_row"] == 1 and info["resident_ctas"] == (2 if grid == "ORCA025" else 1) * sm_count(), info
    assert_psi_close(got, k2_ref(m.e1v, m.e3v_0, ib, rec, cfg), grid)


# ---- bin tiers on adversarial (T, S) ------------------------------------------------------------------------------------
def default_binning(pref, eos):
    nbins, smin, sstp = oracle.default_bins(pref, eos == 2)
    return (pref, eos, smin, sstp, nbins)


BINNINGS = [default_binning(p, e) for p, e in ((0.0, 0), (1000.0, 0), (2000.0, 0), (0.0, 1), (2000.0, 1), (0.0, 2))]
CUSTOM = [(0.0, 0, 23.0, 0.05, 1), (0.0, 0, 45.0, 0.05, 60)]   # one bin; sigmin above the data


def ref_bins(t, s, cfg, sps=0.0):
    pref, eos, smin, sstp, nbins = cfg
    with np.errstate(all="ignore"):
        return npo.mocsig_bins(t, s, F4(sps), pref, eos, smin, sstp, nbins)[0]


def edge_cells(cfg):
    """For T on a grid over -2..34 degC and every interior bin edge: the adjacent float32 salinities between which the
    reference bin changes (bisection over the bit patterns), widened by 3 ulps on each side -> (t, s) float32."""
    nbins = cfg[4]
    tg, bg = np.meshgrid(np.linspace(-1.9, 33.9, 19).astype(F4), np.arange(2, nbins + 1))
    tt, bb = tg.ravel(), bg.ravel()
    lo = np.full(tt.shape, F4(1.0).view(np.int32), np.int64)
    hi = np.full(tt.shape, F4(45.0).view(np.int32), np.int64)
    bits = lambda x: x.astype(np.int32).view(F4)
    ok = (ref_bins(tt, bits(lo), cfg) < bb) & (ref_bins(tt, bits(hi), cfg) >= bb)
    tt, bb, lo, hi = tt[ok], bb[ok], lo[ok], hi[ok]
    while (hi - lo > 1).any():
        mid = (lo + hi) // 2
        up = ref_bins(tt, bits(mid), cfg) >= bb
        hi, lo = np.where(up, mid, hi), np.where(up, lo, mid)
    assert np.all(ref_bins(tt, bits(lo), cfg) < ref_bins(tt, bits(hi), cfg))
    s = np.concatenate([bits(lo + d) for d in range(-3, 5)])
    return np.tile(tt, 8), s


def odd_cells():
    """The tier-1 domain box edges +-1 ulp, zero / missing / negative / large salinities, and non-finite, huge,
    subnormal and signed-zero values in T and in S."""
    up = lambda x: np.nextafter(F4(x), F4(np.inf))
    dn = lambda x: np.nextafter(F4(x), F4(-np.inf))
    box_t = [f(x) for x in (-4.0, 42.0) for f in (dn, F4, up)]
    box_s = [f(x) for x in (1.0, 45.0) for f in (dn, F4, up)]
    special = [F4(x) for x in (np.nan, np.inf, -np.inf, 1e30, -1e30, 1e-40, -1e-40, -0.0, 0.0)]
    t = box_t + [F4(10.0)] * len(box_s) + [F4(10.0)] * 5 + special + [F4(10.0)] * len(special)
    s = [F4(35.0)] * len(box_t) + box_s + [F4(x) for x in (0.0, 9999.0, -5.0, 60.0, -1e-3)] + [F4(35.0)] * len(special) + special
    tc, sc = np.meshgrid(np.array(special, F4), np.array(special, F4))
    return np.concatenate([np.array(t, F4), tc.ravel()]), np.concatenate([np.array(s, F4), sc.ravel()])


@pytest.fixture(scope="module")
def adversarial_ts():
    parts = [edge_cells(cfg) for cfg in BINNINGS] + [odd_cells()]
    return {"edges": parts[:-1], "odd": parts[-1]}


def gpu_bins_stats(t, s, cfg, spt=0.0, sps=0.0):
    """cdfmocsig_bins_device on a 1 x n grid -> (bins, (cells, cells past tier 1, cells on the reference chain))."""
    n = t.size
    pref, eos, smin, sstp, nbins = cfg
    lib.cdfmocsig_setup(np.ones((1, n), F4), np.ones((2, 1, n), F4), np.ones((1, n, 1), np.int16), 2, nbins, smin, sstp,
                        pref, eos, 0.0, spt, sps)
    d_t, d_s = torch.from_numpy(t.reshape(1, 1, n)).cuda(), torch.from_numpy(s.reshape(1, 1, n)).cuda()
    d_b = torch.empty((1, 1, n), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    stats = lib.cdfmocsig_bins_device_stats(d_t, d_s, d_b)
    lib.synchronize()
    return d_b.cpu().numpy().reshape(-1), stats


def test_k2_bin_tiers_diagnostic_kernel(adversarial_ts):
    """Cells on every interior edge of the six default binnings (and box-edge / odd values) through the production bin
    function: equal to the numpy oracle bit for bit under every binning, with tiers 2 and 3 provably reached."""
    t = np.concatenate([p[0] for p in adversarial_ts["edges"]] + [adversarial_ts["odd"][0]])
    s = np.concatenate([p[1] for p in adversarial_ts["edges"]] + [adversarial_ts["odd"][1]])
    for cfg in BINNINGS + CUSTOM:
        got, (n, past1, slow) = gpu_bins_stats(t, s, cfg)
        ref = ref_bins(t, s, cfg)
        assert n == t.size
        assert np.array_equal(got, ref), (cfg, int((got != ref).sum()))
        print(f"bins {cfg}: {n} cells, tier 2 {past1 - slow}, tier 3 {slow}")
        if cfg in BINNINGS[:5]:
            assert lib.cdfmocsig_filter_info()["tier1"] and past1 - slow > 0 and slow > 0, (cfg, n, past1, slow)
    # missing values: the kernel scrubs T == spt and S == sps to 0 before the bin, as the reference does
    t2, s2 = t.copy(), s.copy()
    t2[::11], s2[5::13] = F4(-999.0), F4(9999.0)
    got, _ = gpu_bins_stats(t2, s2, BINNINGS[0], spt=-999.0, sps=9999.0)
    scrub = lambda a, sp: np.where(a == F4(sp), F4(0.0), a).astype(F4)
    assert np.array_equal(got, ref_bins(scrub(t2, -999.0), scrub(s2, 9999.0), BINNINGS[0], sps=9999.0))


@pytest.mark.parametrize("grid,which", [("ORCA2", 0), ((1442, 24, 75), 2)], ids=["orca2-sigma0", "1442x24x75-sigma2000"])
def test_k2_bin_tiers_fused(monkeypatch, adversarial_ts, grid, which):
    """The edge cells of one binning (and the odd values) scattered over wet cells of a record, mixed with ordinary ones
    in the same windows: the default plan, CDFGPU_K2_TIER1=0 and CDFGPU_EXACT_EOS=1 give the same bits, and the oracle."""
    m = synth.make_mesh(grid)
    ib = case_inputs(oracle, m, synth)[0]
    v, t, s = (np.ascontiguousarray(a).copy() for a in mesh_k2(m, 82))
    et, es = adversarial_ts["edges"][which]
    ot, os_ = adversarial_ts["odd"]
    ct, cs = np.concatenate([et, ot]), np.concatenate([es, os_])
    rng = np.random.default_rng(83)
    wet = np.flatnonzero(m.tmask[:-1].reshape(-1))
    assert ct.size <= wet.size // 2
    pos = rng.choice(wet, ct.size, replace=False)
    t.reshape(-1)[pos], s.reshape(-1)[pos] = ct, cs
    cfg = BINNINGS[which]
    runs = {}
    for name, knobs in (("default", {}), ("tier1 off", {"CDFGPU_K2_TIER1": 0}), ("exact eos", {"CDFGPU_EXACT_EOS": 1})):
        set_knobs(monkeypatch, K2_KNOBS, knobs)
        runs[name] = k2_run(m.e1v, m.e3v_0, ib, m.nz, cfg, [(v, t, s)])[0]
        info = lib.cdfmocsig_filter_info()
        assert info["tier1"] == (name == "default") and info["tier2"] == (name != "exact eos"), (name, info)
    for name, o in runs.items():
        assert np.array_equal(o, runs["default"], equal_nan=True), f"{name} differs from the default plan"
    assert_psi_close(runs["default"], k2_ref(m.e1v, m.e3v_0, ib, (v, t, s), cfg), f"{grid}")
