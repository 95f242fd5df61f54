"""K1 skips the area loads of 16-byte vectors whose four area words are +0.0f (land: e3m is already x vmask).  The skip is
exact by construction; these cases pin the places where it could go wrong: non-finite V on zero-area cells, vectors that
straddle row / level ends and the end of the array, -0.0 areas, an area field rebuilt by -vvl, and the batched launch."""
import numpy as np
import pytest

from cdftools_b200 import synth
from util import assert_psi_close, case_inputs

pytestmark = pytest.mark.gpu


def land_mesh(oracle_mod, nx, ny, nz, seed=7):
    """Synthetic mesh with land at both ends of every row, at the last cells of the array and on the whole last level read
    (k = nz-2), so that the flat vectors straddle wet / dry row and level boundaries."""
    m = synth.make_mesh((nx, ny, nz), seed=synth.SEED + seed)
    ib, e3m = case_inputs(oracle_mod, m, synth)
    e3m = e3m.copy()
    e3m[:, :, :2] = 0.0
    e3m[:, :, -3:] = 0.0
    e3m[nz - 2] = 0.0
    e3m[nz - 3, -1, nx // 2:] = 0.0
    return m, ib, e3m


def records(m, n, first=0):
    return [np.ascontiguousarray(synth.make_v_record(m, first + r, adversarial=(r % 2 == 1))[:-1]) for r in range(n)]


def device_single_and_batch(lib, e1v, e3m, ib, recs):
    """Every record once through cdfmoc_gpu_compute_device and once in one cdfmoc_gpu_compute_device_batch launch; the two
    must agree bit for bit (NaN where NaN).  -> the per-record results."""
    import torch
    nz, ny, nb = lib.cdfmoc_setup(e1v, e3m, ib)
    d = [torch.from_numpy(r).cuda() for r in recs]
    single = torch.full((len(recs), nz, ny, nb), 7.0, dtype=torch.float64, device="cuda")
    batch = torch.full_like(single, -7.0)
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(st):
        for r in range(len(recs)):
            lib.cdfmoc_compute_device(d[r], single[r], st)
        lib.cdfmoc_compute_device_batch(d, [batch[r] for r in range(len(recs))], st)
    st.synchronize()
    s, b = single.cpu().numpy(), batch.cpu().numpy()
    assert np.array_equal(s, b, equal_nan=True)
    return s


def check(lib, oracle_mod, e1v, e3m, ib, recs, what):
    got = device_single_and_batch(lib, e1v, e3m, ib, recs)
    for r, v in enumerate(recs):
        with np.errstate(all="ignore"):
            ref = oracle_mod.cdfmoc_record(e1v, e3m, ib, v)
        assert_psi_close(got[r], ref, f"{what} rec {r}")
    return got


@pytest.mark.parametrize("nx,ny,nz", [(37, 11, 6), (182, 23, 7), (1442, 9, 5)])
def test_k1_zero_area_widths(gpu_lib, oracle_mod, nx, ny, nz):
    m, ib, e3m = land_mesh(oracle_mod, nx, ny, nz)
    assert (e3m[: nz - 1] == 0).mean() > 0.2 and (e3m[: nz - 1] != 0).any()
    check(gpu_lib, oracle_mod, m.e1v, e3m, ib, records(m, 4), f"nx={nx}")


@pytest.mark.parametrize("nx,ny,nz", [(37, 11, 6), (182, 23, 7), (1442, 9, 5)])
def test_k1_nonfinite_v_on_zero_area_cells(gpu_lib, oracle_mod, nx, ny, nz):
    """NaN / +Inf / -Inf where the area is zero (land, the dry last level, the last cell of the array) poison their (j,k)
    rows exactly as in the reference, although those area words are never read."""
    m, ib, e3m = land_mesh(oracle_mod, nx, ny, nz)
    recs = records(m, 3)
    v = recs[0]
    v[1, 2, 0] = np.nan                 # land at the row start
    v[2, 4, nx - 1] = np.inf            # land at the row end
    v[nz - 2, 3, 5] = -np.inf           # the fully dry level
    v[nz - 2, ny - 1, nx - 1] = np.nan  # last cell of the array
    dry = np.argwhere(e3m[: nz - 1] == 0)
    k, j, i = dry[len(dry) // 2]
    recs[1][k, j, i] = np.inf
    assert e3m[1, 2, 0] == 0 and e3m[2, 4, nx - 1] == 0 and e3m[nz - 2, 3, 5] == 0 and e3m[nz - 2, ny - 1, nx - 1] == 0
    got = check(gpu_lib, oracle_mod, m.e1v, e3m, ib, recs, "non-finite on land")
    assert np.isnan(got[0][1, 2]).all() and np.isnan(got[0][nz - 2, ny - 1]).all()
    assert np.isnan(got[1][k, j]).all() and not np.isnan(got[2]).any()


def test_k1_signed_zero_area(gpu_lib, oracle_mod):
    """An area of exactly -0.0 (e1v = -0.0 in one column) is not zero for the bitmap; a dry column between wet ones is."""
    nx, ny, nz = 182, 17, 6
    m, ib, e3m = land_mesh(oracle_mod, nx, ny, nz)
    e1v = m.e1v.copy()
    e1v[:, 61] = -0.0
    e3m[:, :, 90] = 0.0
    assert (e3m[: nz - 2, :, 89] != 0).any() and (e3m[: nz - 2, :, 91] != 0).any()
    recs = records(m, 3)
    recs[0][0, 3, 61] = np.nan           # -0.0 * NaN: the row is poisoned
    recs[0][1, 5, 90] = -np.inf          # dry column between wet ones
    got = check(gpu_lib, oracle_mod, e1v, e3m, ib, recs, "signed zeros")
    assert np.isnan(got[0][0, 3]).all() and np.isnan(got[0][1, 5]).all()


def test_k1_vvl_bitmap_follows_the_area(gpu_lib, oracle_mod):
    """cdfmoc_gpu_set_e3v with a thickness field that wets dry cells and dries wet ones: the skip follows the new area."""
    nx, ny, nz = 182, 19, 7
    m, ib, e3m = land_mesh(oracle_mod, nx, ny, nz)
    e3b = (e3m * np.float32(1.0625)).astype(np.float32)
    e3b[:, :, :2] = 9.5                  # dry row starts become wet
    e3b[nz - 2, : ny // 2] = 12.25       # half of the dry last level becomes wet
    e3b[0, 3:9, 20:120] = 0.0            # wet cells become dry
    v = records(m, 2, first=11)
    nz_, ny_, nb = gpu_lib.cdfmoc_setup(m.e1v, e3m, ib)
    out = np.empty((nz, ny, nb))
    gpu_lib.cdfmoc_submit(0, 0, v[1])
    gpu_lib.cdfmoc_fetch(0, out)
    assert_psi_close(out, oracle_mod.cdfmoc_record(m.e1v, e3m, ib, v[1]), "before -vvl")
    gpu_lib.cdfmoc_set_e3v(e3b)
    gpu_lib.cdfmoc_submit(1, 1, v[1])
    gpu_lib.cdfmoc_fetch(1, out)
    assert_psi_close(out, oracle_mod.cdfmoc_record(m.e1v, e3b, ib, v[1]), "after -vvl")
    v[0][0, 5, 50] = np.nan              # wet before, dry now: still poisons the row
    gpu_lib.cdfmoc_submit(2, 2, v[0])
    gpu_lib.cdfmoc_fetch(2, out)
    with np.errstate(all="ignore"):
        ref = oracle_mod.cdfmoc_record(m.e1v, e3b, ib, v[0])
    assert np.isnan(ref[0, 5]).all()
    assert_psi_close(out, ref, "after -vvl, NaN on a dried cell")


def test_k1_no_land(gpu_lib, oracle_mod):
    """An all-wet mesh: no area load is skipped."""
    m = synth.make_mesh((182, 21, 6))
    ib, _ = case_inputs(oracle_mod, m, synth)
    e3m = np.ascontiguousarray(m.e3v_0, dtype=np.float32)
    assert (e3m != 0).all()
    recs = [np.ascontiguousarray(synth.make_v_record(m, r, adversarial=True)[:-1]) for r in range(3)]
    check(gpu_lib, oracle_mod, m.e1v, e3m, ib, recs, "no land")


def test_k1_orca2_batch_equals_single(gpu_lib, oracle_mod):
    """Batched and per-record launches agree bit for bit on a real-shaped mesh with land."""
    m = synth.make_mesh("ORCA2")
    ib, e3m = case_inputs(oracle_mod, m, synth)
    check(gpu_lib, oracle_mod, m.e1v, e3m, ib, records(m, 5), "ORCA2")
