"""K1 applies the basin masks once per flat 16-byte vector (its lead byte) and adds the in-row cells with another non-zero
byte -- the row's exceptions -- cell by cell, one lane each; a row with more than 32 takes the literal chain.  These cases
pin where that could go wrong: two or three bytes in every vector of a row (more exceptions than a warp has lanes),
exceptions at the first and last cell of a row for every width mod 4, eight basins (the whole byte), NaN / Inf V on
exception, byte-0 and out-of-row cells, exceptions on dry levels, and an area rebuilt by -vvl.  Every case is checked
against the C oracle, and single-record and batched launches must agree bit for bit."""
import numpy as np
import pytest

from cdftools_b200 import synth
from test_gpu_k1_zero_area import check, records
from util import assert_psi_close

pytestmark = pytest.mark.gpu


def masks_from_bytes(byt, nb):
    """(ny, nx) basin bytes -> ibmask (ny, nx, nb) INTEGER(2) of 0 / 1."""
    return np.ascontiguousarray(((byt[:, :, None].astype(np.int32) >> np.arange(nb)) & 1).astype(np.int16))


def wet_e3m(m):
    """e3v without land: cells of byte 0 are wet too, so their V meets a non-zero area."""
    return np.ascontiguousarray(m.e3v_0[: m.nz], dtype=np.float32).copy()


def halo_bytes(nx, ny, seed):
    """ORCA-like bytes: global + one sub-basin inside, the global bit cleared on the halo columns i = 0 and nx-1 (as
    cdfmoc.f90:325-336 does), patches of land (byte 0) and a second sub-basin on some rows."""
    rng = np.random.default_rng(seed)
    byt = np.full((ny, nx), 0b00011, np.uint8)
    byt[ny // 2:, :] = 0b10101
    byt[:, 0] &= 0b11110
    byt[:, nx - 1] &= 0b11110
    land = rng.random((ny, nx)) < 0.15
    byt[land] = 0
    byt[1, :] = 0b00011                         # a row whose only exceptions are its two ends
    byt[1, 0], byt[1, nx - 1] = 0b00010, 0b00010
    return byt


@pytest.mark.parametrize("nx", [181, 182, 183, 184])
def test_k1_exceptions_at_row_ends(gpu_lib, oracle_mod, nx):
    """Exceptions at i = 0 and i = nx-1 for every nx mod 4: odd ny makes every row shift s occur over the levels."""
    ny, nz = 7, 6
    m = synth.make_mesh((nx, ny, nz), seed=synth.SEED + nx)
    ib = masks_from_bytes(halo_bytes(nx, ny, nx), 5)
    e3m = wet_e3m(m)
    e3m[1, :, : nx // 3] = 0.0                 # dry cells, the first column included
    check(gpu_lib, oracle_mod, m.e1v, e3m, ib, records(m, 3), f"row ends nx={nx}")


def test_k1_more_exceptions_than_lanes(gpu_lib, oracle_mod):
    """Bytes cycling 3, 5, 21, 3 along a row (two exceptions per vector, ~90 per row: the literal chain), basins
    alternating every cell (~90 per row too) and random bytes (rows of up to 32 exceptions and beyond)."""
    nx, ny, nz = 182, 9, 5
    m = synth.make_mesh((nx, ny, nz), seed=synth.SEED + 3)
    rng = np.random.default_rng(3)
    byt = np.array([0b00011, 0b00101, 0b10101, 0b00011], np.uint8)[np.arange(nx) % 4][None, :].repeat(ny, axis=0)
    byt[2:4] = np.where(np.arange(nx) % 2 == 0, 0b00011, 0b00101)
    byt[4:] = rng.choice(np.array([0, 1, 2, 3, 12, 13, 20, 21, 31], np.uint8), size=(ny - 4, nx))
    ib = masks_from_bytes(byt, 5)
    check(gpu_lib, oracle_mod, m.e1v, wet_e3m(m), ib, records(m, 3), "alternating basins")


@pytest.mark.parametrize("nx", [37, 1442])
def test_k1_eight_basins(gpu_lib, oracle_mod, nx):
    """NB = 8: the lead byte uses all eight bits; mostly 255 with 128, 1 and land mixed in."""
    ny, nz = 11, 5
    m = synth.make_mesh((nx, ny, nz), seed=synth.SEED + 8)
    rng = np.random.default_rng(8)
    byt = rng.choice(np.array([255, 255, 255, 255, 255, 128, 1, 0, 0x81], np.uint8), size=(ny, nx))
    ib = masks_from_bytes(byt, 8)
    check(gpu_lib, oracle_mod, m.e1v, wet_e3m(m), ib, records(m, 3), f"eight basins nx={nx}")


def test_k1_nonfinite_v_on_exception_byte0_and_out_of_row_cells(gpu_lib, oracle_mod):
    """NaN / Inf V on exception cells of one and of two other bytes, a byte-0 cell and on the last cell of a row, which
    the first vector of the next row holds as an out-of-row cell (nx = 182: row (k, j) starts 2 cells into its vector
    when k*ny + j is odd): each poisons its own row and only that row; also on such cells of a dry level."""
    nx, ny, nz = 182, 7, 6
    m = synth.make_mesh((nx, ny, nz), seed=synth.SEED + 5)
    byt = halo_bytes(nx, ny, 5)
    byt[2, 40:44] = [0b00011, 0b00101, 0b00011, 0b00011]   # i = 41: an exception of its vector
    byt[2, 82:86] = [0b00011, 0b00101, 0b00011, 0b10101]   # level 1 (s = 2): i = 83 and 85 are exceptions
    byt[3, 60] = 0
    byt[4, 98:106] = [0b10101, 0b10101, 0b10101, 0b00011, 0b10101, 0b10101, 0b00011, 0b00101]   # level 3 (s = 2): i = 101,
    # 104 and 105 are exceptions
    ib = masks_from_bytes(byt, 5)
    e3m = wet_e3m(m)
    e3m[3, 4, :] = 0.0                          # a dry level of row 4
    recs = records(m, 3)
    v = recs[0]
    v[0, 2, 41] = np.nan                        # exception cell
    recs[2][1, 2, 85] = np.inf                  # exception cell
    v[1, 3, 60] = np.inf                        # byte-0 cell
    v[2, 2, nx - 1] = -np.inf                   # last cell of row (2, 2), held by the first vector of row (2, 3)
    v[3, 4, 101] = np.nan                       # exception cell on the dry level
    recs[2][3, 4, 105] = -np.inf                # exception cell on the dry level
    recs[1][2, 4, nx - 1] = np.nan              # last cell of row (2, 4), held by the first vector of row (2, 5)
    got = check(gpu_lib, oracle_mod, m.e1v, e3m, ib, recs, "non-finite V")
    for k, j in ((0, 2), (1, 3), (2, 2), (3, 4)):
        assert not np.isfinite(got[0][k, j]).any()
    assert not np.isfinite(got[2][1, 2]).any() and not np.isfinite(got[2][3, 4]).any()
    assert np.isfinite(got[0][2:, 3]).all() and np.isfinite(got[1][:, 5]).all() and np.isfinite(got[2][4:]).all()


def test_k1_vector_basins_vvl(gpu_lib, oracle_mod):
    """-vvl rebuilds the area, not the mask words or the exception lists: the same mesh before and after
    cdfmoc_gpu_set_e3v."""
    nx, ny, nz = 183, 9, 6
    m = synth.make_mesh((nx, ny, nz), seed=synth.SEED + 6)
    rng = np.random.default_rng(6)
    byt = halo_bytes(nx, ny, 6)
    byt[5:7] = rng.choice(np.array([0, 3, 5, 21], np.uint8), size=(2, nx))
    ib = masks_from_bytes(byt, 5)
    e3m = wet_e3m(m)
    e3b = (e3m * np.float32(1.0625)).astype(np.float32)
    e3b[2, :, ::3] = 0.0                       # exception cells among them become dry
    v = records(m, 2, first=21)
    gpu_lib.cdfmoc_setup(m.e1v, e3m, ib)
    out = np.empty((nz, ny, 5))
    gpu_lib.cdfmoc_submit(0, 0, v[0])
    gpu_lib.cdfmoc_fetch(0, out)
    assert_psi_close(out, oracle_mod.cdfmoc_record(m.e1v, e3m, ib, v[0]), "before -vvl")
    gpu_lib.cdfmoc_set_e3v(e3b)
    for r in range(2):
        gpu_lib.cdfmoc_submit(1, 1, v[r])
        gpu_lib.cdfmoc_fetch(1, out)
        assert_psi_close(out, oracle_mod.cdfmoc_record(m.e1v, e3b, ib, v[r]), f"after -vvl rec {r}")
