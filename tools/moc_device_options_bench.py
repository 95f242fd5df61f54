"""cdfmoc -decomp, cdfmocsig -isodep and the cdfmaxmoc windows on device-resident records, ORCA025 L75, one GPU; and the
-decomp results and shear-pass time of another build of the library (the parent commit's) beside this one.

    python tools/moc_device_options_bench.py --out FILE [--parent-lib variants/libcdfgpu_parent.so] [--calls N]

Every timed call reads records resident beyond L2: two records of V, T, S (3 x 436 MB each) used in turn, after a warm-up.
  * decomp_device: N calls on a torch stream, CUDA events on that stream, per call = window / N (best of three windows);
    launches per call from cdfgpu_launch_count.
  * the host path: decomp_submit + decomp_fetch of the same records from pageable numpy arrays, host clock (median of N).
  * compute_device_isodep against compute_device (sigma0, 104 classes): plain K2 without -isodep, and with it.
  * one maxmoc_device call over 12 windows against 12 cdfmoc_gpu_maxmoc slot calls (host clock, both synchronised).
  * with --parent-lib, in child processes alternating parent / this build three times: the shear pass's kernel time per
    record (sum of the zsig0 and geostrophic-recurrence kernels in a torch.profiler trace of decomp_submit) and the
    launches per record; and the four -decomp slabs of both builds on seeded ORCA025 L75 records and random edge shapes,
    compared bit for bit (this build also through decomp_device).
The GPU's name and power limit are read in the same run.  Needs a GPU: there is no CPU fallback.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

KEYS = ("total", "sh", "bt", "ag")
SHEAR = ("decomp_sigma_kernel", "decomp_geo_level_kernel", "decomp_geo_column_kernel")
EDGE_SHAPES = [(37, 9, 6), (1, 5, 4), (2, 6, 4), (9, 1, 4), (9, 2, 4), (37, 9, 2), (40, 12, 76)]


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or ["?, ?"])[0].split(",", 1)
    return {"gpu": name.strip(), "power_limit": power.strip()}


def orca025_case():
    import oracle
    from cdftools_b200 import synth
    from test_gpu_moc_option_edges import mesh_case, mesh_record
    oracle.build()
    m = synth.make_mesh("ORCA025")
    return m, mesh_case(m), [mesh_record(m, 100 + r) for r in range(2)]


def setup(lib, c):
    shape = lib.cdfmoc_setup(c.e1v, c.e3m, c.ib)
    lib.cdfmoc_decomp_setup(c.e1u, c.gphiv, c.gdept, c.um, c.tm, teos10=c.teos10)
    return shape


# ---- child processes: one build of the library each (CDFGPU_LIB) ------------------------------------------------------------
def load_any_build():
    """lib with only the entry points this build exports declared: an older build lacks the device calls added since."""
    import ctypes
    from cdftools_b200 import lib
    so = ctypes.CDLL(str(lib.SO_PATH))
    for name in [n for n in lib.SIGNATURES if not hasattr(so, n)]:
        del lib.SIGNATURES[name]
    return lib


def child_shear(out):
    """Shear-pass kernel time and launches per record of decomp_submit, ORCA025 L75."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    lib = load_any_build()
    lib.init(0, 3)
    _, c, recs = orca025_case()
    shape = setup(lib, c)
    recs = [tuple(np.ascontiguousarray(a) for a in r) for r in recs]
    for r in range(2):
        lib.cdfmoc_decomp_submit(0, r, *recs[r])
        lib.cdfmoc_decomp_fetch(0, shape)
    n0, nrec = lib.launch_count(), 6
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for r in range(nrec):
            lib.cdfmoc_decomp_submit(0, r, *recs[r % 2])
            lib.cdfmoc_decomp_fetch(0, shape)
        torch.cuda.synchronize()
    launches = (lib.launch_count() - n0) / nrec
    us = {}
    for e in prof.events():
        for k in SHEAR:
            if k in e.name:
                t = getattr(e, "device_time", None) or getattr(e, "cuda_time", 0.0)
                us[k] = us.get(k, 0.0) + t
    json.dump({"shear_ms_per_record": sum(us.values()) / nrec / 1e3,
               "by_kernel_ms_per_record": {k: v / nrec / 1e3 for k, v in us.items()},
               "launches_per_record": launches}, open(out, "w"))


def child_parity(out):
    """The four slabs of decomp_submit (and of decomp_device when the build has it) on the seeded cases -> npz."""
    import torch
    from test_gpu_moc_option_edges import random_case
    lib = load_any_build()
    lib.init(0, 3)
    has_device = "cdfmoc_gpu_decomp_device" in lib.SIGNATURES
    _, c, recs = orca025_case()
    cases = [("orca025", c, recs)]
    for nx, ny, nz in EDGE_SHAPES:
        c, rec = random_case(nx, ny, nz, 3, 7 * nx + ny + nz)
        cases.append((f"random_{nx}x{ny}x{nz}", c, [rec]))
    res = {}
    for name, c, recs in cases:
        shape = setup(lib, c)
        for r, rec in enumerate(recs):
            rec = tuple(np.ascontiguousarray(a) for a in rec)
            lib.cdfmoc_decomp_submit(0, r, *rec)
            got = lib.cdfmoc_decomp_fetch(0, shape)
            for k in KEYS:
                res[f"{name}/{r}/submit/{k}"] = got[k]
            if has_device:
                src = [torch.from_numpy(a).cuda() for a in rec]
                o = [torch.empty(shape, dtype=torch.float64, device="cuda") for _ in KEYS]
                torch.cuda.synchronize()
                lib.cdfmoc_decomp_device(*src, *o)
                lib.synchronize()
                for k, t in zip(KEYS, o):
                    res[f"{name}/{r}/device/{k}"] = t.cpu().numpy()
    np.savez(out, **res)


def run_child(what, libpath, out):
    env = dict(os.environ)
    if libpath:
        env["CDFGPU_LIB"] = str(libpath)
    subprocess.run([sys.executable, __file__, "--child", what, "--out", str(out)], check=True, env=env, cwd=ROOT)


# ---- this build's device calls ------------------------------------------------------------------------------------------------
def events_per_call(fn, st, calls):
    import torch
    best = float("inf")
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for n in range(calls):
            fn(n)
        e1.record(st)
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1) / calls)
    return best


def measure_this(calls):
    import oracle
    import torch
    from cdftools_b200 import lib, synth
    from util import case_inputs
    lib.init(0, 3)
    m, c, recs = orca025_case()
    shape = setup(lib, c)
    st = torch.cuda.Stream()
    d = [[torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in r] for r in recs]
    o = [torch.empty(shape, dtype=torch.float64, device="cuda") for _ in KEYS]
    torch.cuda.synchronize()
    dec = lambda n: lib.cdfmoc_decomp_device(*d[n % 2], *o, stream=st)
    for n in range(4):
        dec(n)
    st.synchronize()
    n0 = lib.launch_count()
    dec(0)
    st.synchronize()
    out = {"decomp_device_launches": lib.launch_count() - n0}
    out["decomp_device_ms"] = events_per_call(dec, st, calls)
    host = [tuple(np.ascontiguousarray(a) for a in r) for r in recs]
    ts = []
    for n in range(calls):
        t0 = time.perf_counter()
        lib.cdfmoc_decomp_submit(0, n, *host[n % 2])
        lib.cdfmoc_decomp_fetch(0, shape)
        ts.append(time.perf_counter() - t0)
    out["decomp_submit_fetch_ms_median"] = 1e3 * float(np.median(ts))

    # cdfmaxmoc: 12 windows on one slab -- the whole slab and a box for every basin, one cell, the closed southern rows
    wins = [(b, 1, m.ny, 1, m.nz) for b in range(5)] + [(b, 600, 900, 10, 60) for b in range(5)] + [(1, 700, 700, 20, 20),
                                                                                                   (0, 1, 3, 1, m.nz)]
    lib.cdfmoc_maxmoc_windows(wins)
    ovt = torch.empty((12, 2), dtype=torch.float32, device="cuda")
    loc = torch.empty((12, 4), dtype=torch.int32, device="cuda")
    lib.cdfmoc_submit(1, 0, host[0][0])
    lib.cdfmoc_fetch(1, np.empty(shape))
    lib.cdfmoc_compute_device(d[0][0], o[0], st)
    mx = lambda n: lib.cdfmoc_maxmoc_device(o[0], ovt, loc, stream=st)
    for n in range(3):
        mx(n)
    st.synchronize()
    ts, ts1 = [], []
    for n in range(calls):
        t0 = time.perf_counter()
        mx(n)
        st.synchronize()
        t1 = time.perf_counter()
        for w in wins:
            lib.cdfmoc_maxmoc(1, *w)
        ts.append(t1 - t0)
        ts1.append(time.perf_counter() - t1)
    out["maxmoc_device_12_windows_ms_median"] = 1e3 * float(np.median(ts))
    out["maxmoc_slot_12_calls_ms_median"] = 1e3 * float(np.median(ts1))
    out["maxmoc_device_12_windows_event_ms"] = events_per_call(mx, st, calls)
    lib.cdfmoc_teardown()

    # cdfmocsig sigma0 / 104 classes
    ib = case_inputs(oracle, m, synth)[0]
    sshape = lib.cdfmocsig_setup(m.e1v, m.e3v_0, ib, m.nz, 104, 23.0, 0.05, 0.0, 0)
    so = [torch.empty(sshape, dtype=torch.float64, device="cuda") for _ in range(2)]
    torch.cuda.synchronize()
    plain = lambda n: lib.cdfmocsig_compute_device(d[n % 2][0], d[n % 2][1], d[n % 2][2], so[0], stream=st)
    for n in range(4):
        plain(n)
    out["mocsig_compute_device_ms"] = events_per_call(plain, st, calls)
    st.synchronize()
    lib.cdfmocsig_set_isodep(m.gdept_1d)
    iso = lambda n: lib.cdfmocsig_compute_device_isodep(d[n % 2][0], d[n % 2][1], d[n % 2][2], so[0], so[1], stream=st)
    for n in range(4):
        iso(n)
    out["mocsig_compute_device_isodep_ms"] = events_per_call(iso, st, calls)
    for n in range(4):
        plain(n)
    out["mocsig_compute_device_with_isodep_on_ms"] = events_per_call(plain, st, calls)
    st.synchronize()
    lib.finalize()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--child", default=None)
    a = ap.parse_args()
    if a.child == "shear":
        return child_shear(a.out)
    if a.child == "parity":
        return child_parity(a.out)
    res = {"case": "ORCA025 L75 (1442 x 1021 x 75), 5 basins, synthetic seeded records", **card()}
    res["this_build"] = measure_this(a.calls)
    if a.parent_lib:
        with tempfile.TemporaryDirectory() as tmp:
            runs = []
            for rep in range(3):
                for tag, libpath in (("parent", a.parent_lib), ("new", None)):
                    f = Path(tmp) / f"shear_{tag}_{rep}.json"
                    run_child("shear", libpath, f)
                    runs.append({"build": tag, **json.loads(f.read_text())})
            res["shear_pass_alternating"] = runs
            for tag, libpath in (("parent", a.parent_lib), ("new", None)):
                run_child("parity", libpath, Path(tmp) / f"parity_{tag}.npz")
            p, n = np.load(Path(tmp) / "parity_parent.npz"), np.load(Path(tmp) / "parity_new.npz")
            same = lambda x, y: x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8))
            differ = [k for k in p.files if not same(p[k], n[k])]
            differ += [k for k in n.files if "/device/" in k and not same(n[k], n[k.replace("/device/", "/submit/")])]
            res["parity"] = {"slabs_compared": len(p.files) + sum("/device/" in k for k in n.files),
                             "cases": sorted({k.split("/")[0] for k in p.files}), "bitwise_differences": differ}
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    sys.exit(main())
