"""The record-input settings of the library: the byte-order flag (cdfgpu_set_input_big_endian) is one process-wide value that
cdfgpu_finalize resets for every device, and every call decodes its record arrays with exactly the kernels its declarations
ask for (K3 swap, K3b unpack), counted with cdfgpu_launch_count."""
import numpy as np
import pytest

from cdftools_b200 import synth
from test_gpu_packed import PACK, SP, decoded, ts_records, v_records
from test_gpu_sibling_inputs import TRANSIG_KINDS, reset_siblings, transig_frames
from util import case_inputs

pytestmark = pytest.mark.gpu


def reset(lib):
    """Every record-input setting at its default: host-order REAL(4) everywhere."""
    reset_siblings(lib)
    for f in range(5):
        lib.set_input_packing(f, lib.INPUT_F32)
    lib.set_input_big_endian(False)


@pytest.fixture
def lib(gpu_lib):
    reset(gpu_lib)
    yield gpu_lib
    reset(gpu_lib)


def swapped(a):
    """The raw big-endian file bytes of a host-order array."""
    return np.ascontiguousarray(a.byteswap())


def launches(lib, call):
    n0 = lib.launch_count()
    call()
    return lib.launch_count() - n0


def test_finalize_resets_the_byte_order_of_every_device(lib, oracle_mod):
    """A byte order set before a one-device session is gone after cdfgpu_finalize on every device, so a later two-device
    session reads host-order records on both devices alike (odd slots run on the second device)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    m = synth.make_mesh("SMALL")
    ib, e3m = case_inputs(oracle_mod, m, synth)
    nrec = 6
    vs = [synth.make_v_record(m, r, adversarial=(r % 2 == 1))[:-1] for r in range(nrec)]

    def run_all():
        ns = lib.nslots()
        shape = lib.cdfmoc_setup(m.e1v, e3m, ib)
        out = np.empty((nrec,) + shape)
        for r0 in range(0, nrec, ns):
            idx = range(r0, min(nrec, r0 + ns))
            for r in idx:
                lib.cdfmoc_submit(r % ns, r, vs[r])
            for r in idx:
                lib.cdfmoc_fetch(r % ns, out[r])
        lib.cdfmoc_teardown()
        return out

    one = run_all()
    lib.set_input_big_endian(True)
    lib.finalize()
    try:
        lib.init_multi(2, "time", 3)
        assert lib.nslots() == nrec
        two = run_all()
    finally:
        lib.finalize()
        lib.init(0, 3)
    assert np.abs(one).max() > 0
    assert np.array_equal(one, two)


def test_submit_launches(lib, oracle_mod):
    m = synth.make_mesh("SMALL")
    ib, e3m = case_inputs(oracle_mod, m, synth)
    shape = lib.cdfmoc_setup(m.e1v, e3m, ib)
    raw = v_records(m, 1)[0]
    v = decoded(raw, "v")
    out = np.empty(shape)

    def moc(zv):
        n = launches(lib, lambda: lib.cdfmoc_submit(0, 0, zv))
        lib.cdfmoc_fetch(0, out)
        return n

    assert moc(v) == 1             # K1
    lib.set_input_big_endian(True)
    assert moc(swapped(v)) == 2    # K3 swap, K1
    lib.set_input_big_endian(False)
    lib.set_input_packing(0, lib.INPUT_I16, *PACK["v"], SP)
    assert moc(raw) == 2           # K3b unpack, K1
    lib.cdfmoc_teardown()

    lib.cdfmocsig_setup(m.e1v, m.e3v_0, synth.setup_masks(m), m.nz, 158, 30.0, 0.05, 2000.0, lib.EOS80, float(SP), float(SP),
                        float(SP))
    t, s = ts_records(m, 1)[0]
    for f, kind in enumerate(("v", "t", "s")):
        lib.set_input_packing(f, lib.INPUT_I16, *PACK[kind], SP)
    assert launches(lib, lambda: lib.cdfmocsig_submit(0, 0, raw, t, s)) == 4   # three K3b unpacks, K2
    lib.cdfmocsig_fetch(0, np.empty((m.ny, 158, 5)))
    lib.cdfmocsig_teardown()


def test_sibling_launches_under_the_process_byte_order(lib, oracle_mod):
    """With cdfgpu_set_input_big_endian on and no field declared, cdfzonal_gpu_sum swaps nothing and cdftransig_gpu_record
    swaps each of its four fields."""
    m = synth.make_mesh("SMALL")
    lib.set_input_big_endian(True)
    nk = m.nz - 1
    msk = m.vmask[:nk].astype(np.float32)
    shape = lib.cdfzonal_setup(m.e1v, m.e1v, oracle_mod.zonal_masks(msk[0]), msk)
    zv = synth.make_v_record(m, 0)[:nk]
    assert launches(lib, lambda: lib.cdfzonal_sum(zv, shape)) == 1   # K4
    lib.cdfzonal_teardown()

    pref, nb, smin, scal, zoom, smn = lib.TRANSIG_CODES["1000"]
    _, _, itab, step = lib.transig_bins(nb, smin, scal, zoom, smn)
    fr = [decoded(a, kind) for a, kind in zip(transig_frames(m, 1)[0], TRANSIG_KINDS)]
    e2u = (m.e1u * np.float32(0.9)).astype(np.float32)
    lib.cdftransig_setup(e2u, m.e1v, fr[4], fr[5], m.nz, nb, pref, smin, step, itab)
    rec = [swapped(a) for a in fr[:4]]
    assert launches(lib, lambda: lib.cdftransig_record(*rec, set_masks=True)) == 2 + 4   # four K3 swaps, K6 density, K6 scatter
    lib.cdftransig_teardown()
