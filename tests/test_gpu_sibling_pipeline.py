"""The record pipelines of the sibling tools (cdfzonal_gpu_submit_* / cdfmhst_gpu_submit* / cdftransig_gpu_submit and their
fetch / wait): bit for bit what the synchronous calls give, with the field declarations read at submit, the buffer contract,
the error codes, the launch counts, time sharding over several devices, and the command-line twins on more records than
slots."""
import os

import numpy as np
import pytest
from scipy.io import netcdf_file

from cdftools_b200 import build, ncfiles, synth
from test_gpu_packed import decoded, quantize
from test_gpu_sibling_inputs import (MHST_OUTS, TRANSIG_KINDS, declare, handed, reset_siblings, run_cli, stored, transig_frames,
                                     vts_records, write_nc)

pytestmark = pytest.mark.gpu
NAN = float("nan")
ERR_ARG, ERR_STATE = 2, 3


def reset(lib):
    reset_siblings(lib)
    for f in range(5):
        lib.set_input_packing(f, lib.INPUT_F32)
    lib.set_input_big_endian(False)


@pytest.fixture
def lib(gpu_lib):
    reset(gpu_lib)
    yield gpu_lib
    reset(gpu_lib)
    gpu_lib.finalize()          # back to the session's context: one device, three slots
    gpu_lib.init(0, 3)


def session(lib, nslots, ndev=1):
    lib.finalize()
    if ndev == 1:
        lib.init(0, nslots)
    else:
        lib.init_multi(ndev, "time", nslots)


def two_gpus(lib):
    if lib.device_count() < 2:
        pytest.skip("needs two GPUs")


def same(a, b):
    if isinstance(a, tuple):
        return len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    if a is None or b is None:
        return a is None and b is None
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


def pipeline(lib, n, submit, fetch):
    """Records 0..n-1 through slots r mod nslots(), a slot's record fetched right before the slot is reused; results in
    record order."""
    ns = lib.nslots()
    out = [None] * n
    for r in range(n):
        if r >= ns:
            out[r - ns] = fetch((r - ns) % ns)
        submit(r % ns, r)
    for r in range(max(0, n - ns), n):
        out[r] = fetch(r % ns)
    return out


def raises(code, fn, *a, **k):
    from cdftools_b200 import lib as L
    with pytest.raises(L.CdfGpuError) as e:
        fn(*a, **k)
    assert e.value.code == code, e.value


# ---- cases ------------------------------------------------------------------------------------------------------------------
def zonal_case(lib, oracle_mod, grid="ODD", nk=None):
    m = synth.make_mesh(grid)
    nk = m.nz - 1 if nk is None else nk
    msk = m.vmask[:nk].astype(np.float32)
    zm = oracle_mod.zonal_masks(msk[0], m.tmaskatl, m.tmaskind, m.tmaskpac)
    e2 = (m.e1v * np.float32(0.75)).astype(np.float32)
    shape = lib.cdfzonal_setup(m.e1v, e2, zm, msk)
    alpha = (0.5 + np.arange(m.ny) / m.ny).astype(np.float32)
    return m, nk, shape, alpha


def zonal_records(m, nk, n):
    recs = [quantize(synth.make_v_record(m, r, adversarial=(r % 3 == 1))[:nk], "v", m.vmask[:nk] == 0) for r in range(n)]
    return recs


# the three zonal calls a record may go through: sum, sum with alpha, mean with the max / min
def zonal_sync(lib, kind, zv, shape, alpha):
    if kind == 0:
        return lib.cdfzonal_sum(zv, shape)
    if kind == 1:
        return lib.cdfzonal_sum(zv, shape, alpha)
    return lib.cdfzonal_mean(zv, shape, 99999.0, True)


def zonal_submit(lib, kind, slot, zv, alpha):
    if kind == 2:
        lib.cdfzonal_submit_mean(slot, zv, 99999.0, True)
    else:
        lib.cdfzonal_submit_sum(slot, zv, alpha if kind == 1 else None)


def mhst_case(lib, m):
    return lib.cdfmhst_setup(m.e1v, m.e3v_0, m.vmask[0].astype(np.float32), m.tmaskatl, m.tmaskpac, m.tmaskind)


def mhst_records(m, n):
    recs = []
    for r in range(n):
        v, t, s = (decoded(a, k) for a, k in zip(vts_records(m, r), ("v", "t", "s")))
        if r % 2 == 1:   # non-finite cells
            t[2, 5, 7], t[3, 6, 9], s[1, 4, 11], v[4, 8, 12] = NAN, np.inf, -np.inf, np.inf
        recs.append((v, t, s))
    return recs


def transig_case(lib, m, vvl):
    pref, nb, smin, scal, zoom, smn = lib.TRANSIG_CODES["1000"]
    _, _, itab, step = lib.transig_bins(nb, smin, scal, zoom, smn)
    e2u = (m.e1u * np.float32(0.9)).astype(np.float32)
    frames = transig_frames(m, 7)
    e3 = (None, None) if vvl else (decoded(frames[0][4], "e3"), decoded(frames[0][5], "e3"))
    lperio = bool(m.glamv[0, 0] == m.glamv[0, m.nx - 2])
    return lambda: lib.cdftransig_setup(e2u, m.e1v, *e3, m.nz, nb, pref, smin, step, itab, lperio=lperio), frames


def transig_args(fr, reps, vvl):
    nf = 6 if vvl else 4
    arg = [handed(fr[a], TRANSIG_KINDS[a], reps[a]) for a in range(nf)]
    return arg[:4], dict(e3u_vvl=arg[4] if vvl else None, e3v_vvl=arg[5] if vvl else None)


def transig_pipeline(lib, setup, frames, vvl, reps_of=lambda r: ("f32",) * 6, nslots=None, refill=False):
    """The frames through the frame pipeline (two tags: the first half sets the masks), each frame declared as reps_of(r)
    says right before its submit; refill: the slot's arrays are overwritten with NaN right after its wait returns."""
    shape = setup()
    ns = nslots or lib.load().cdfgpu_nslots() // max(lib.num_devices(), 1)
    held = [None] * ns
    for r, fr in enumerate(frames):
        slot = r % ns
        if r >= ns:
            lib.cdftransig_wait(slot)
            if refill:
                for a in held[slot][0] + [x for x in held[slot][1].values() if x is not None]:
                    a.view(np.uint8)[:] = 0xFF
        reps = reps_of(r)
        for a in range(6):
            declare(lib, lib.CALL_TRANSIG, a, reps[a], TRANSIG_KINDS[a])
        held[slot] = transig_args(fr, reps, vvl)
        lib.cdftransig_submit(slot, *held[slot][0], set_masks=r < len(frames) // 2, **held[slot][1])
    out = lib.cdftransig_fetch(shape)
    lib.cdftransig_teardown()
    return out


def transig_sync(lib, setup, frames, vvl):
    shape = setup()
    reset_siblings(lib)
    for r, fr in enumerate(frames):
        a, k = transig_args(fr, ("f32",) * 6, vvl)
        lib.cdftransig_record(*a, set_masks=r < len(frames) // 2, **k)
    out = lib.cdftransig_fetch(shape)
    lib.cdftransig_teardown()
    return out


# ---- 1. pipeline = synchronous -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nslots", [1, 3, 8])
@pytest.mark.parametrize("grid", ["ODD", "2d"])
def test_zonal_pipeline_equals_synchronous(lib, oracle_mod, nslots, grid):
    session(lib, nslots)
    m, nk, shape, alpha = zonal_case(lib, oracle_mod, "ODD", 1 if grid == "2d" else None)
    n = 2 * nslots + 1
    recs = [decoded(a, "v") for a in zonal_records(m, nk, n)]
    ref = [zonal_sync(lib, r % 3, recs[r], shape, alpha) for r in range(n)]
    assert np.abs(ref[0]).max() > 0
    got = pipeline(lib, n, lambda s, r: zonal_submit(lib, r % 3, s, recs[r], alpha), lambda s: lib.cdfzonal_fetch(s, shape))
    for r in range(n):
        assert same(got[r], ref[r]), r
    assert lib.cdfzonal_kernel_ms() > 0
    lib.cdfzonal_teardown()


@pytest.mark.parametrize("nslots", [1, 3, 8])
@pytest.mark.parametrize("zdim", [False, True])
def test_mhst_pipeline_equals_synchronous(lib, nslots, zdim):
    session(lib, nslots)
    m = synth.make_mesh("SMALL")
    dims = mhst_case(lib, m)
    n = 2 * nslots + 1
    recs = mhst_records(m, n)
    # even records: -vt mode on the V-point products; odd records: V, T, S with NaN / Inf cells
    prods = [(v * t, v * s) for v, t, s in recs]
    ref = [lib.cdfmhst_record(*prods[r], dims, zdim) if r % 2 == 0 else lib.cdfmhst_record_vts(*recs[r], dims, zdim)
           for r in range(n)]
    assert any(np.isnan(h).any() for h, _ in ref[1::2])

    def submit(s, r):
        if r % 2 == 0:
            lib.cdfmhst_submit(s, *prods[r], zdim)
        else:
            lib.cdfmhst_submit_vts(s, *recs[r], zdim)

    got = pipeline(lib, n, submit, lambda s: lib.cdfmhst_fetch(s, dims))
    for r in range(n):
        assert same(got[r], ref[r]), r
    assert lib.cdfmhst_kernel_ms() > 0
    lib.cdfmhst_teardown()


@pytest.mark.parametrize("nslots", [1, 3, 8])
@pytest.mark.parametrize("vvl", [False, True])
def test_transig_pipeline_equals_synchronous(lib, nslots, vvl):
    session(lib, nslots)
    m = synth.make_mesh("SMALL")
    setup, frames = transig_case(lib, m, vvl)
    frames = (frames * 3)[:2 * nslots + 1]
    ref = transig_sync(lib, setup, frames, vvl)
    assert np.abs(ref[0]).max() > 0 and np.abs(ref[1]).max() > 0
    got = transig_pipeline(lib, setup, frames, vvl, nslots=nslots)
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])


# ---- 2. declarations are read at submit ----------------------------------------------------------------------------------
def test_declarations_are_captured_at_submit(lib, oracle_mod):
    m, nk, shape, alpha = zonal_case(lib, oracle_mod)
    raws = zonal_records(m, nk, 7)
    ref = [lib.cdfzonal_sum(decoded(a, "v"), shape, alpha) for a in raws]
    reps = ("f32", "f32be", "i16be")
    held = {}

    def submit(s, r):   # the declaration changes between submits of records that are in flight together
        declare(lib, lib.CALL_ZONAL, 0, reps[r % 3], "v")
        held[s] = handed(raws[r], "v", reps[r % 3])
        lib.cdfzonal_submit_sum(s, held[s], alpha)

    got = pipeline(lib, len(raws), submit, lambda s: lib.cdfzonal_fetch(s, shape))
    for r in range(len(raws)):
        assert same(got[r], ref[r]), (r, reps[r % 3])
    lib.cdfzonal_teardown()
    reset_siblings(lib)

    dims = mhst_case(lib, m)
    recs = [vts_records(m, r) for r in range(5)]
    ref = [lib.cdfmhst_record_vts(*(decoded(a, k) for a, k in zip(rec, ("v", "t", "s"))), dims) for rec in recs]

    def submit_vts(s, r):
        rr = [reps[(r + f) % 3] for f in range(3)]
        for f, kind in enumerate(("v", "t", "s")):
            declare(lib, lib.CALL_MHST_VTS, f, rr[f], kind)
        lib.cdfmhst_submit_vts(s, *(handed(a, k, rep) for a, k, rep in zip(recs[r], ("v", "t", "s"), rr)))

    got = pipeline(lib, len(recs), submit_vts, lambda s: lib.cdfmhst_fetch(s, dims))
    for r in range(len(recs)):
        assert same(got[r], ref[r]), r
    lib.cdfmhst_teardown()
    reset_siblings(lib)

    m = synth.make_mesh("SMALL")
    for vvl in (False, True):
        setup, frames = transig_case(lib, m, vvl)
        ref = transig_sync(lib, setup, frames, vvl)
        all_reps = ("f32", "f32be", "i16", "i16be")
        got = transig_pipeline(lib, setup, frames, vvl, lambda r: tuple(all_reps[(r + a) % 4] for a in range(6)))
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), vvl


# ---- 3. buffer contract ---------------------------------------------------------------------------------------------------
def test_refilling_a_slot_after_its_fetch_or_wait_changes_nothing(lib, oracle_mod):
    m, nk, shape, alpha = zonal_case(lib, oracle_mod)
    recs = [decoded(a, "v") for a in zonal_records(m, nk, 7)]
    ref = [lib.cdfzonal_sum(z, shape, alpha) for z in recs]
    ns = lib.nslots()
    bufs = [lib.PinnedArray(recs[0].shape) for _ in range(ns)]
    out = [None] * len(recs)
    for r, z in enumerate(recs):
        s = r % ns
        if r >= ns:
            out[r - ns] = lib.cdfzonal_fetch(s, shape)
            bufs[s].array[:] = np.nan           # refilled right after the fetch returns
        bufs[s].array[:] = z
        lib.cdfzonal_submit_sum(s, bufs[s].array, alpha)
    for r in range(len(recs) - ns, len(recs)):
        out[r] = lib.cdfzonal_fetch(r % ns, shape)
        bufs[r % ns].array[:] = np.nan
    for r in range(len(recs)):
        assert same(out[r], ref[r]), r
    for b in bufs:
        b.free()
    lib.cdfzonal_teardown()

    m = synth.make_mesh("SMALL")
    for vvl in (False, True):
        setup, frames = transig_case(lib, m, vvl)
        ref = transig_sync(lib, setup, frames, vvl)
        got = transig_pipeline(lib, setup, frames, vvl, refill=True)
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), vvl


# ---- 4. errors ----------------------------------------------------------------------------------------------------------
def test_pipeline_errors(lib, oracle_mod):
    m, nk, shape, alpha = zonal_case(lib, oracle_mod, "TINY")
    z = decoded(zonal_records(m, nk, 1)[0], "v")
    ns = lib.nslots()
    for slot in (-1, ns):
        raises(ERR_ARG, lib.cdfzonal_submit_sum, slot, z)
        raises(ERR_ARG, lib.cdfzonal_submit_mean, slot, z)
        raises(ERR_ARG, lib.cdfzonal_fetch, slot, shape)
        raises(ERR_ARG, lib.cdfmhst_fetch, slot, (m.nz, m.ny))
    raises(ERR_STATE, lib.cdfzonal_fetch, 1, shape)             # never submitted
    lib.cdfzonal_submit_sum(1, z)
    raises(ERR_STATE, lib.cdfzonal_sum, z, shape)               # a record in flight
    raises(ERR_STATE, lib.cdfzonal_mean, z, shape)
    raises(ERR_STATE, lib.cdfzonal_submit_sum, 1, z)            # the slot's record has not been fetched
    got = lib.cdfzonal_fetch(1, shape)
    raises(ERR_STATE, lib.cdfzonal_fetch, 1, shape)             # fetched already
    ref = lib.cdfzonal_sum(z, shape)
    assert same(got, ref)
    lib.cdfzonal_submit_sum(2, z)
    shape = lib.cdfzonal_setup(*zonal_setup_args(oracle_mod, m, nk))   # setup waits and forgets the record
    raises(ERR_STATE, lib.cdfzonal_fetch, 2, shape)
    assert same(lib.cdfzonal_sum(z, shape), ref)
    lib.cdfzonal_submit_sum(0, z)
    lib.cdfzonal_teardown()
    raises(ERR_STATE, lib.cdfzonal_fetch, 0, shape)

    dims = mhst_case(lib, m)
    v, t, s = mhst_records(m, 1)[0]
    raises(ERR_STATE, lib.cdfmhst_fetch, 0, dims)
    lib.cdfmhst_submit_vts(ns - 1, v, t, s)
    raises(ERR_STATE, lib.cdfmhst_record, v * t, v * s, dims)
    raises(ERR_STATE, lib.cdfmhst_record_vts, v, t, s, dims)
    lib.cdfmhst_fetch(ns - 1, dims)
    lib.cdfmhst_submit(0, v * t, v * s)
    mhst_case(lib, m)
    raises(ERR_STATE, lib.cdfmhst_fetch, 0, dims)
    lib.cdfmhst_submit(0, v * t, v * s)
    lib.cdfmhst_teardown()
    raises(ERR_STATE, lib.cdfmhst_fetch, 0, dims)

    setup, frames = transig_case(lib, synth.make_mesh("SMALL"), False)
    tshape = setup()
    a, k = transig_args(frames[0], ("f32",) * 6, False)
    raises(ERR_ARG, lib.cdftransig_submit, ns, *a, set_masks=True)
    raises(ERR_ARG, lib.cdftransig_wait, -1)
    raises(ERR_ARG, lib.cdftransig_wait, ns)
    raises(ERR_STATE, lib.cdftransig_wait, 0)
    lib.cdftransig_submit(1, *a, set_masks=True)
    raises(ERR_STATE, lib.cdftransig_record, *a, set_masks=True)
    lib.cdftransig_wait(1)
    raises(ERR_STATE, lib.cdftransig_wait, 1)
    lib.cdftransig_record(*a, set_masks=True)
    lib.cdftransig_submit(2, *a, set_masks=True)
    lib.cdftransig_fetch(tshape)                                # drains every frame
    raises(ERR_STATE, lib.cdftransig_wait, 2)
    lib.cdftransig_submit(0, *a, set_masks=True)
    setup()
    raises(ERR_STATE, lib.cdftransig_wait, 0)
    lib.cdftransig_teardown()
    raises(ERR_STATE, lib.cdftransig_wait, 0)


def zonal_setup_args(oracle_mod, m, nk):
    msk = m.vmask[:nk].astype(np.float32)
    return m.e1v, (m.e1v * np.float32(0.75)).astype(np.float32), oracle_mod.zonal_masks(msk[0], m.tmaskatl, m.tmaskind, m.tmaskpac), msk


# ---- 5. launch counts ---------------------------------------------------------------------------------------------------
def launches(lib, call):
    n0 = lib.launch_count()
    call()
    return lib.launch_count() - n0


def test_submit_launches_equal_the_synchronous_calls(lib, oracle_mod):
    m, nk, shape, alpha = zonal_case(lib, oracle_mod, "TINY")
    raw = zonal_records(m, nk, 1)[0]
    for rep in ("f32", "f32be", "i16"):
        declare(lib, lib.CALL_ZONAL, 0, rep, "v")
        z = handed(raw, "v", rep)
        sync = launches(lib, lambda: lib.cdfzonal_sum(z, shape))
        assert sync == (1 if rep == "f32" else 2)
        assert launches(lib, lambda: lib.cdfzonal_submit_sum(2, z)) == sync
        lib.cdfzonal_fetch(2, shape)
    lib.cdfzonal_teardown()
    reset_siblings(lib)
    dims = mhst_case(lib, m)
    v, t, s = mhst_records(m, 1)[0]
    assert launches(lib, lambda: lib.cdfmhst_record(v, t, dims)) == 1
    assert launches(lib, lambda: lib.cdfmhst_submit(1, v, t)) == 1
    lib.cdfmhst_fetch(1, dims)
    assert launches(lib, lambda: lib.cdfmhst_record_vts(v, t, s, dims)) == 2
    assert launches(lib, lambda: lib.cdfmhst_submit_vts(1, v, t, s)) == 2
    lib.cdfmhst_fetch(1, dims)
    lib.cdfmhst_teardown()
    setup, frames = transig_case(lib, synth.make_mesh("SMALL"), False)
    setup()
    lib.set_input_big_endian(True)
    a = [np.ascontiguousarray(x.byteswap()) for x in transig_args(frames[0], ("f32",) * 6, False)[0]]
    assert launches(lib, lambda: lib.cdftransig_record(*a, set_masks=True)) == 6
    assert launches(lib, lambda: lib.cdftransig_submit(1, *a, set_masks=True)) == 6
    lib.cdftransig_wait(1)
    lib.cdftransig_teardown()


# ---- 6. two devices --------------------------------------------------------------------------------------------------------
def test_time_sharded_siblings_are_bit_identical_and_use_both_devices(lib, oracle_mod):
    two_gpus(lib)
    import torch
    grid = (1442, 200, 12)   # a slot holds 12 MB of record on its device
    m, nk, shape, alpha = zonal_case(lib, oracle_mod, grid)
    recs = [decoded(a, "v") for a in zonal_records(m, nk, 9)]
    ref = [zonal_sync(lib, r % 3, recs[r], shape, alpha) for r in range(9)]
    dims = mhst_case(lib, m)
    mrec = mhst_records(m, 5)
    mref = [lib.cdfmhst_record_vts(*x, dims) for x in mrec]
    tset, frames = transig_case(lib, synth.make_mesh("SMALL"), True)
    tref = transig_sync(lib, tset, frames, True)
    session(lib, 3, ndev=2)
    assert lib.num_devices() == 2 and lib.nslots() == 6
    zonal_case(lib, oracle_mod, grid)
    free0 = torch.cuda.mem_get_info(1)[0]
    got = pipeline(lib, 9, lambda s, r: zonal_submit(lib, r % 3, s, recs[r], alpha), lambda s: lib.cdfzonal_fetch(s, shape))
    assert free0 - torch.cuda.mem_get_info(1)[0] >= 2 * recs[0].nbytes   # slots 1, 3, 5 allocated on the second device
    assert all(same(a, b) for a, b in zip(got, ref))
    assert same(lib.cdfzonal_sum(recs[0], shape), ref[0])
    mhst_case(lib, m)
    got = pipeline(lib, 5, lambda s, r: lib.cdfmhst_submit_vts(s, *mrec[r]), lambda s: lib.cdfmhst_fetch(s, dims))
    assert all(same(a, b) for a, b in zip(got, mref))
    got = transig_pipeline(lib, tset, frames, True, nslots=3)
    assert np.array_equal(got[0], tref[0]) and np.array_equal(got[1], tref[1])
    lib.cdfzonal_teardown()
    lib.cdfmhst_teardown()


# ---- 7. command-line twins: more records than slots ----------------------------------------------------------------------
@pytest.fixture(scope="module")
def tools():
    return build.build_host()


def zonal_files(m, d, nrec, how):
    v3 = [quantize(synth.make_v_record(m, r, adversarial=(r % 2 == 1)), "v", m.vmask == 0) for r in range(nrec)]
    v2 = [quantize(synth.make_ts_record(m, r)[0][0], "t", m.tmask[0] == 0) for r in range(nrec)]
    write_nc(d / "in.nc", m, "depthv", nrec, {"vomecrty": stored(v3, "v", how), "sosstsst": stored(v2, "t", how)})
    return v3, v2


def test_cli_zonal_records_beyond_the_slots(tools, oracle_mod, tmp_path):
    m = synth.make_mesh("ORCA2")
    nrec = 7
    d = {how: tmp_path / how for how in ("packed", "float")}
    for how in d:
        ncfiles.write_mesh(m, d[how])
        v3, v2 = zonal_files(m, d[how], nrec, how)
        run_cli(tools["cdfzonalsum_gpu"], ["-f", "in.nc", "-p", "V", "-b", "new_maskglo.nc"], d[how])
        run_cli(tools["cdfzonalmean_gpu"], ["-f", "in.nc", "-p", "V", "-b", "new_maskglo.nc", "-max"], d[how])
    for out in ("zonalsum.nc", "zonalmean.nc"):
        assert (d["packed"] / out).read_bytes() == (d["float"] / out).read_bytes(), out
    e2 = (m.e1v * np.float32(0.75)).astype(np.float32)
    msk = m.vmask.astype(np.float32)
    zm = oracle_mod.zonal_masks(msk[0], m.tmaskatl, m.tmaskind, m.tmaskpac)
    dl = oracle_mod.zonal_dlsurf(m.e1v, e2)
    f = netcdf_file(str(d["float"] / "zonalsum.nc"), "r", mmap=False)
    g = netcdf_file(str(d["float"] / "zonalmean.nc"), "r", mmap=False)
    assert f.variables["zoimecrty_glo"].shape[0] == nrec
    for r in range(nrec):
        z3, z2 = decoded(v3[r], "v"), decoded(v2[r], "t")
        ref3 = oracle_mod.zonalsum_record(zm, msk, z3, dl)
        ref2 = oracle_mod.zonalsum_record(zm, msk[:1], z2[None], dl)
        _, zmax, zmin = oracle_mod.zonalmean_record(zm, msk, z3, dl, 0.0, True)
        for b, sfx in enumerate(["_glo", "_atl", "_inp", "_ind", "_pac"]):
            assert np.allclose(f.variables["zoimecrty" + sfx][r, :, :, 0], ref3[b].astype(np.float32), rtol=3e-7,
                               atol=1e-3 * np.abs(ref3).max() * 1e-7), (r, sfx)
            assert np.allclose(f.variables["zoisstsst" + sfx][r, :, 0], ref2[b, 0].astype(np.float32), rtol=3e-7,
                               atol=1e-3 * np.abs(ref2).max() * 1e-7), (r, sfx)
            assert np.array_equal(g.variables["zomecrty" + sfx + "_max"][r, :, :, 0], zmax[b])
            assert np.array_equal(g.variables["zomecrty" + sfx + "_min"][r, :, :, 0], zmin[b])
    f.close()
    g.close()


def mhst_files(m, d, nrec, how):
    recs = [vts_records(m, r) for r in range(nrec)]
    write_nc(d / "gridV.nc", m, "depthv", nrec, {"vomecrty": stored([r[0] for r in recs], "v", how)})
    write_nc(d / "gridT.nc", m, "deptht", nrec, {"votemper": stored([r[1] for r in recs], "t", how, "_FillValue")})
    write_nc(d / "gridS.nc", m, "deptht", nrec, {"vosaline": stored([r[2] for r in recs], "s", how, "_FillValue")})
    return recs


def test_cli_mhst_records_beyond_the_slots(tools, oracle_mod, tmp_path):
    from test_gpu_host_e2e import _mhst_expected
    from test_gpu_sibling_inputs import vpoint
    m = synth.make_mesh("SMALL")
    nrec = 6
    d = {how: tmp_path / how for how in ("packed", "float", "oracle")}
    for how in ("packed", "float"):
        ncfiles.write_mesh(m, d[how])
        mhst_files(m, d[how], nrec, how)
        run_cli(tools["cdfmhst_gpu"], ["-v", "gridV.nc", "-t", "gridT.nc", "-s", "gridS.nc", "-MST"], d[how])
    for out in MHST_OUTS:
        assert (d["packed"] / out).read_bytes() == (d["float"] / out).read_bytes(), out
    ncfiles.write_mesh(m, d["oracle"])   # the files of tests/test_gpu_host_e2e.py::test_cdfmhst_cli_separate_files, more records
    vrec = ncfiles.write_gridv(m, d["oracle"] / "gridV.nc", nrec)
    trec = ncfiles.write_gridt(m, d["oracle"] / "gridT.nc", nrec)
    run_cli(tools["cdfmhst_gpu"], ["-v", "gridV.nc", "-t", "gridT.nc", "-MST"], d["oracle"])
    f = netcdf_file(str(d["oracle"] / "mhst.nc"), "r", mmap=False)
    for r in range(nrec):
        ref = _mhst_expected(oracle_mod, m, *vpoint(vrec[r], trec[r][0], trec[r][1]), True, False)
        for name, exp in ref.items():
            got = f.variables[name][r, :, :, 0]
            filled = exp == np.float32(9999.99)
            assert np.array_equal(got == np.float32(9999.99), filled), (r, name)
            assert np.allclose(got[~filled], exp[~filled], rtol=3e-7, atol=1e-30), (r, name)
    f.close()
    txt = (d["oracle"] / "zonal_heat_trp.dat").read_text()
    assert [int(l.split()[-1]) for l in txt.splitlines() if "time :" in l] == list(range(1, nrec + 1))


def transig_files(m, d, frames, how, tags):
    full = lambda a: np.concatenate([a, a[-1:]])
    per = len(frames) // len(tags)
    for t, tag in enumerate(tags):
        fr = frames[per * t:per * t + per]
        pre = str(d / f"SYN-B200_{tag}_grid")
        write_nc(pre + "U.nc", m, "depthu", per, {"vozocrtx": stored([full(f[0]) for f in fr], "v", how)})
        write_nc(pre + "V.nc", m, "depthv", per, {"vomecrty": stored([full(f[1]) for f in fr], "v", how)})
        write_nc(pre + "T.nc", m, "deptht", per, {"votemper": stored([full(f[2]) for f in fr], "t", how, "_FillValue")})
        write_nc(pre + "S.nc", m, "deptht", per, {"vosaline": stored([full(f[3]) for f in fr], "s", how, "_FillValue")})


TAGS = ("y2026m01", "y2026m02", "y2026m03")


def test_cli_transig_frames_beyond_the_slots(tools, oracle_mod, tmp_path):
    m = synth.make_mesh("SMALL")
    d = {how: tmp_path / how for how in ("packed", "float", "oracle")}
    for how in ("packed", "float"):
        ncfiles.write_mesh(m, d[how])
        transig_files(m, d[how], transig_frames(m, 6), how, TAGS)
        run_cli(tools["cdftransig_xy3d_gpu"], ["-c", "SYN-B200", "-l", *TAGS, "-S", "-o", "uv.nc"], d[how])
    assert (d["packed"] / "uv.nc").read_bytes() == (d["float"] / "uv.nc").read_bytes()
    # the files of tests/test_gpu_host_e2e.py::test_cdftransig_cli_matches_oracle, three tags of two frames
    ncfiles.write_mesh(m, d["oracle"])
    frames = []
    for t, tag in enumerate(TAGS):
        us = ncfiles.write_gridu(m, d["oracle"] / f"SYN-B200_{tag}_gridU.nc", 2, first=2 * t)
        vs = ncfiles.write_gridv(m, d["oracle"] / f"SYN-B200_{tag}_gridV.nc", 2, first=2 * t)
        ts = ncfiles.write_gridt(m, d["oracle"] / f"SYN-B200_{tag}_gridT.nc", 2, first=2 * t)
        frames += [(us[r], vs[r], ts[r][0], ts[r][1], t == 0) for r in range(2)]
    run_cli(tools["cdftransig_xy3d_gpu"], ["-c", "SYN-B200", "-l", *TAGS, "-o", "uv.nc"], d["oracle"])
    pref, nb, smin, scal, zoom, smn = 1000.0, 93, 24.2, 0.10, 32.3, 0.05
    _, _, itab, scm = oracle_mod.transig_bins(nb, smin, scal, zoom, smn)
    du, dv = np.zeros((nb, m.ny, m.nx)), np.zeros((nb, m.ny, m.nx))
    mu, mv = np.zeros((m.nz - 1, m.ny, m.nx), np.uint8), np.zeros((m.nz - 1, m.ny, m.nx), np.uint8)
    e2u = (m.e1u * np.float32(0.9)).astype(np.float32)
    e3u = (m.e3v_0 * np.float32(1.01)).astype(np.float32)
    lperio = bool(m.glamv[0, 0] == m.glamv[0, m.nx - 2])
    for zu, zv, zt, zs, first in frames:
        oracle_mod.transig_record(e2u, m.e1v, e3u[:-1], m.e3v_0[:-1], zu[:-1], zv[:-1], zt[:-1], zs[:-1], pref, smin, scm, itab, nb,
                                  du, dv, mu, mv, first, lperio)
    f = netcdf_file(str(d["oracle"] / "uv.nc"), "r", mmap=False)
    assert f.variables["vovxysig"].iweight == len(frames)
    for name, ref in (("vouxysig", du), ("vovxysig", dv)):
        got, want = f.variables[name][0], (ref / len(frames)).astype(np.float32)
        assert np.array_equal(got != 0, want != 0), name
        assert np.allclose(got, want, rtol=2e-7, atol=1e-6), (name, np.abs(got - want).max())
    f.close()


def test_cli_two_devices_write_the_same_files(lib, tools, tmp_path):
    two_gpus(lib)
    m = synth.make_mesh("SMALL")
    frames = transig_frames(m, 6)
    for ndev in ("1", "2"):
        d = tmp_path / ndev
        ncfiles.write_mesh(m, d)
        zonal_files(m, d, 7, "packed")
        mhst_files(m, d, 6, "float")
        transig_files(m, d, frames, "packed", TAGS)
    env = dict(os.environ, CDFGPU_SHARD="time")
    import subprocess
    for ndev in ("1", "2"):
        e = dict(env, CDFGPU_DEVICES=ndev)
        for tool, args in (("cdfzonalmean_gpu", ["-f", "in.nc", "-p", "V", "-b", "new_maskglo.nc", "-max"]),
                           ("cdfmhst_gpu", ["-v", "gridV.nc", "-t", "gridT.nc", "-s", "gridS.nc", "-MST"]),
                           ("cdftransig_xy3d_gpu", ["-c", "SYN-B200", "-l", *TAGS, "-S", "-o", "uv.nc"])):
            r = subprocess.run([str(tools[tool])] + args, capture_output=True, text=True, cwd=tmp_path / ndev, env=e, timeout=600)
            assert r.returncode == 0, r.stdout + r.stderr
    for out in ["zonalmean.nc", "uv.nc"] + MHST_OUTS:
        assert (tmp_path / "1" / out).read_bytes() == (tmp_path / "2" / out).read_bytes(), out
