"""Raw and 16-bit packed records decoded on the device for the sibling tools, ORCA025 L75, in one process on one GPU.

    python tools/e2e_siblings.py [--out DIR] [--reps N] [--file-records N]

(a) the C ABI, one record per call: cdfzonal_gpu_sum, cdfmhst_gpu_record_vts and cdftransig_gpu_record, each on host-order
    float32, big-endian float32 (K3 swap) and big-endian int16 (K3b unpack) records from pinned buffers, the three kinds
    alternating; a host clock around each call (every call ends in a stream synchronise).  Then, in a traced run of its own,
    the device time of unpack_i16_kernel and mhst_vpoint_kernel (torch.profiler), with their bytes and share of the copy peak.
(b) the command-line twins cdfzonalsum_gpu, cdfmhst_gpu (-v -t -s) and cdftransig_xy3d_gpu (-S) on float and packed files on
    tmpfs, alternating: the "records" phase of $CDFGPU_TIMING; and, as the host baseline, nc3::Reader::read_f32 against
    read_raw of one record of each field involved.
Prints one JSON line (and writes it to DIR/e2e_siblings.json with --out).  Needs a GPU: there is no CPU fallback.
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
sys.path.insert(0, str(ROOT / "tools"))

from e2e_packed import _READ_TIMER, HBM_COPY_PEAK_GBS, card   # noqa: E402

SP = -32768
PACK = {"vozocrtx": (1.0e-4, 0.0), "vomecrty": (1.0e-4, 0.0), "votemper": (1.0e-3, 15.0), "vosaline": (5.0e-4, 35.0)}
FIELDS = ("vozocrtx", "vomecrty", "votemper", "vosaline")
KINDS = ("f32", "f32be", "i16be")


def quantize(x, name, land):
    sf, ao = PACK[name]
    raw = np.clip(np.rint((x.astype(np.float64) - ao) / sf), -32767, 32767).astype(np.int16)
    raw[land] = SP
    return raw


def decode(raw, name):
    """getvar's three masked passes (src/cdfio.F90:1599-1605) in float32, as K3b applies them."""
    sf, ao = (np.float32(c) for c in PACK[name])
    x = raw.astype(np.float32)
    x = np.where(x != SP, x * sf, x).astype(np.float32)
    if ao != 0:
        x = np.where(x != SP, x + ao, x).astype(np.float32)
    return x


def records(m, r):
    """One time frame of the four fields, (nz, ny, nx) int16."""
    from cdftools_b200 import synth
    t, s = synth.make_ts_record(m, r)
    return {"vozocrtx": quantize(synth.make_v_record(m, 500 + r) * m.umask, "vozocrtx", m.umask == 0),
            "vomecrty": quantize(synth.make_v_record(m, r), "vomecrty", m.vmask == 0),
            "votemper": quantize(t, "votemper", m.tmask == 0), "vosaline": quantize(s, "vosaline", m.tmask == 0)}


def abi(lib, m, reps):
    import oracle
    nz, ny, nx = m.e3v_0.shape
    n3 = nz * ny * nx
    raws = records(m, 0)
    bufs = {}
    for kind in KINDS:   # page-locked buffers of what a host reading the file hands over
        for f in FIELDS:
            a = decode(raws[f], f) if kind.startswith("f32") else raws[f]
            p = lib.PinnedArray(a.shape, a.dtype)
            p.array[...] = a.byteswap() if kind.endswith("be") else a
            bufs[kind, f] = p
    msk = m.vmask.astype(np.float32)
    zshape = lib.cdfzonal_setup(m.e1v, m.e1v, oracle.zonal_masks(msk[0], m.tmaskatl, m.tmaskind, m.tmaskpac), msk)
    mdims = lib.cdfmhst_setup(m.e1v, m.e3v_0, msk[0], m.tmaskatl, m.tmaskpac, m.tmaskind)
    pref, nb, smin, scal, zoom, smn = lib.TRANSIG_CODES["1000"]
    _, _, itab, step = lib.transig_bins(nb, smin, scal, zoom, smn)
    lib.cdftransig_setup(m.e1u, m.e1v, m.e3v_0[:-1], m.e3v_0[:-1], nz, nb, pref, smin, step, itab, lperio=True)

    def use(kind):
        for call, names in ((lib.CALL_ZONAL, ("vomecrty",)), (lib.CALL_MHST_VTS, FIELDS[1:]), (lib.CALL_TRANSIG, FIELDS)):
            for fi, f in enumerate(names):
                if kind == "i16be":
                    lib.set_sibling_input(call, fi, lib.INPUT_I16, True, *PACK[f], SP)
                else:
                    lib.set_sibling_input(call, fi, lib.INPUT_F32, kind == "f32be")

    calls = {
        "cdfzonal_gpu_sum": (lambda k: lib.cdfzonal_sum(bufs[k, "vomecrty"].array, zshape), ("vomecrty",), n3),
        "cdfmhst_gpu_record_vts": (lambda k: lib.cdfmhst_record_vts(*(bufs[k, f].array for f in FIELDS[1:]), mdims), FIELDS[1:], n3),
        "cdftransig_gpu_record": (lambda k: lib.cdftransig_record(*(bufs[k, f].array for f in FIELDS), set_masks=True), FIELDS,
                                  n3 - ny * nx),
    }
    results = {}
    ceiling = lib.h2d_probe(bufs["f32", "vomecrty"], reps=6)
    for name, (fn, names, cells) in calls.items():
        t = {k: [] for k in KINDS}
        for kind in KINDS:   # warm-up: staging buffers, module load
            use(kind)
            fn(kind)
        outs = {}
        for _ in range(reps):
            for kind in KINDS:
                use(kind)
                t0 = time.perf_counter()
                outs[kind] = fn(kind)
                t[kind].append(time.perf_counter() - t0)
        res = {"cells_per_field": cells, "fields": len(names)}
        for kind in KINDS:
            nbytes = cells * len(names) * (2 if kind == "i16be" else 4)
            dt = min(t[kind])
            res[kind] = {"ms": dt * 1e3, "ms_all": [x * 1e3 for x in t[kind]], "h2d_bytes": nbytes, "h2d_gbs_effective": nbytes / dt / 1e9}
        if outs["f32"] is not None:   # the three kinds must give the same result (cdftransig accumulates: nothing per call)
            as_list = lambda x: list(x) if isinstance(x, tuple) else [x]
            res["results_identical"] = all(np.array_equal(a, b) for k in KINDS[1:] for a, b in zip(as_list(outs["f32"]), as_list(outs[k])))
        results[name] = res
    out = {"grid": "ORCA025 L75 (%d x %d x %d)" % (nx, ny, nz), "h2d_ceiling_gbs": ceiling, "calls": results}

    try:   # device time of the decode and V-point kernels, from a traced run of its own
        import torch
        from torch.profiler import ProfilerActivity, profile
        use("i16be")
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                calls["cdfzonal_gpu_sum"][0]("i16be")
                calls["cdfmhst_gpu_record_vts"][0]("i16be")
            torch.cuda.synchronize()
        kern = {}
        for name, nbytes in (("unpack_i16_kernel", n3 * 6), ("mhst_vpoint_kernel", n3 * 20)):
            d = [e.device_time for e in prof.events() if name in e.name and e.device_time > 0]   # microseconds
            if d:
                ms = float(np.median(d)) / 1e3
                gbs = nbytes / (ms * 1e-3) / 1e9
                kern[name] = {"ms_per_record_field": ms, "launches": len(d), "bytes": nbytes, "gbs": gbs,
                              "frac_of_copy_peak": gbs / HBM_COPY_PEAK_GBS}
            else:
                kern[name] = "not measured (no such kernel in the trace)"
        out["kernels"] = kern
    except Exception as e:   # the timings above stand without the trace
        out["kernels"] = "not measured (%s)" % e
    use("f32")
    lib.cdfzonal_teardown()
    lib.cdfmhst_teardown()
    lib.cdftransig_teardown()
    for p in bufs.values():
        p.free()
    return out


def write_grid(path, m, zdim, name, recs, packed):
    from scipy.io import netcdf_file
    f = netcdf_file(str(path), "w", version=2)
    f.createDimension("time_counter", None)
    for n, l in (("x", m.nx), ("y", m.ny), (zdim, m.nz)):
        f.createDimension(n, l)
    tc = f.createVariable("time_counter", "d", ("time_counter",))
    v = f.createVariable(name, "h" if packed else "f", ("time_counter", zdim, "y", "x"))
    if packed:
        v.scale_factor, v.add_offset, v.missing_value = np.float32(PACK[name][0]), np.float32(PACK[name][1]), np.int16(SP)
    else:
        v.missing_value = np.float32(SP)
    for r, raw in enumerate(recs):
        tc[r] = 432000.0 * (r + 0.5)
        v[r] = raw if packed else decode(raw, name)
    f.close()


def files(m, nrec):
    from cdftools_b200 import build, ncfiles
    n3 = m.nz * m.ny * m.nx
    grids = {"vozocrtx": ("U", "depthu"), "vomecrty": ("V", "depthv"), "votemper": ("T", "deptht"), "vosaline": ("S", "deptht")}
    cases = {"cdfzonalsum_gpu": ["-f", "gridV.nc", "-p", "V"], "cdfmhst_gpu": ["-v", "gridV.nc", "-t", "gridT.nc", "-s", "gridS.nc"],
             "cdftransig_xy3d_gpu": ["-c", "SYN", "-l", "y2026", "-S"]}
    outs = {"cdfzonalsum_gpu": ["zonalsum.nc"], "cdfmhst_gpu": ["mhst.nc", "zonal_heat_trp.dat"], "cdftransig_xy3d_gpu": ["uvxysig.nc"]}
    out = {"records_per_file": nrec}
    with tempfile.TemporaryDirectory() as bindir, \
            tempfile.TemporaryDirectory(dir="/dev/shm" if Path("/dev/shm").exists() else None) as d:
        tools = build.build_host(bindir=bindir, names=list(cases))
        timer = Path(bindir) / "read_timer"
        (Path(bindir) / "read_timer.cpp").write_text(_READ_TIMER)
        subprocess.run(["g++", "-O2", "-std=c++17", "-pthread", "-ffp-contract=off", "-I", str(ROOT / "cdftools_b200" / "csrc" / "host"),
                        "-o", str(timer), str(Path(bindir) / "read_timer.cpp")], check=True)
        d = Path(d)
        ncfiles.write_mesh(m, d / "mesh")
        recs = [records(m, r) for r in range(nrec)]
        for kind in ("float", "packed"):
            (d / kind).mkdir()
            for mf in (d / "mesh").iterdir():
                (d / kind / mf.name).symlink_to(mf)
            for name, (g, zdim) in grids.items():
                write_grid(d / kind / f"grid{g}.nc", m, zdim, name, [r[name] for r in recs], kind == "packed")
                (d / kind / f"SYN_y2026_grid{g}.nc").symlink_to(d / kind / f"grid{g}.nc")
        del recs
        host = {}   # host side of one record of each field, page cache warm
        for kind in ("float", "packed"):
            for name, (g, _) in grids.items():
                t = subprocess.run([str(timer), str(d / kind / f"grid{g}.nc"), name, str(n3)], capture_output=True, text=True, check=True)
                f32, raw = map(float, t.stdout.split())
                host["%s_%s" % (name, kind)] = {"read_f32_s": f32, "read_raw_s": raw}
        out["host_read_per_record"] = host
        env = dict(os.environ, CDFGPU_TIMING="1")
        rec = {t: {"float": [], "packed": []} for t in cases}
        same = {}
        for it in range(3):
            for tool, args in cases.items():
                for kind in ("float", "packed"):
                    r = subprocess.run([str(tools[tool])] + args, cwd=d / kind, check=True, capture_output=True, text=True, env=env)
                    ph = {l.split()[2]: float(l.split()[3]) for l in r.stderr.splitlines() if l.startswith(tool + ": phase")}
                    if it:   # the first round warms the page cache
                        rec[tool][kind].append(ph["records"])
                same[tool] = all((d / "float" / o).read_bytes() == (d / "packed" / o).read_bytes() for o in outs[tool])
        out["cli_records_phase_s"] = {t: {k: min(v) for k, v in r.items()} for t, r in rec.items()}
        out["cli_records_phase_s_all"] = rec
        out["cli_outputs_byte_identical"] = same
        out["cli_file_bytes"] = {k: sum((d / k / f"grid{g}.nc").stat().st_size for g, _ in grids.values()) for k in ("float", "packed")}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--file-records", type=int, default=2)
    a = ap.parse_args()
    from cdftools_b200 import lib, synth
    res = {"tool": "tools/e2e_siblings.py", **card()}
    m = synth.make_mesh("ORCA025")
    lib.init(0, 3)
    try:
        res["abi"] = abi(lib, m, a.reps)
    finally:
        lib.finalize()
    res["files"] = files(m, a.file_records)
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).mkdir(parents=True, exist_ok=True)
        (Path(a.out) / "e2e_siblings.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
