"""The *_device entry points of the sibling tools against their host-array calls, ORCA025 L75, one process on one GPU.

    python tools/sibling_device_bench.py [--out DIR] [--calls N]

For each case (cdfzonal sum, mean, mean -max; cdfmhst vt, vts; one cdftransig frame):
  * device path: N calls (after a warm-up) on a torch stream over two device-resident records in rotation (each ~440 MB,
    well above the 126 MB L2), timed with CUDA events on that stream; per call = window / N, three windows.
  * host path: the synchronous host-array call on the same record from pinned memory, host clock (best and median of 5), and
    the kernel time inside it (*_kernel_ms).
  * algorithmic bytes as bench.py's siblings() counts them (cdfmhst _vts: K5v's 20 B per cell plus K5's 12 B), achieved GB/s
    of the device path and its share of the 6545.6 GB/s device-to-device copy peak.
The GPU's name and power limit are read in the same run.  Prints one JSON line (and writes DIR/sibling_device.json with
--out).  Needs a GPU: there is no CPU fallback.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

HBM_COPY_PEAK_GBS = 6545.6   # device-to-device copy peak the project measures its kernels against (DESIGN.md section 4)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or ["?, ?"])[0].split(",", 1)
    return {"gpu": name.strip(), "power_limit": power.strip()}


def pinned(lib, a, keep):
    p = lib.PinnedArray(a.shape, a.dtype)
    p.array[...] = a
    keep.append(p)
    return p.array


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--calls", type=int, default=60)
    args = ap.parse_args()
    import torch
    from cdftools_b200 import lib, synth

    lib.init(0, 3)
    m = synth.make_mesh("ORCA025")
    nk, ny, nx = m.nz - 1, m.ny, m.nx
    n3, n3z = nk * ny * nx, m.nz * ny * nx
    keep = []
    st = torch.cuda.Stream()
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()

    def device_ms(call, recs):
        """per-call ms of call(record, stream) over args.calls calls, records in rotation: three windows."""
        with torch.cuda.stream(st):
            for i in range(6):
                call(recs[i % len(recs)], st)
        torch.cuda.synchronize()
        ms = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(st):
                e0.record(st)
                for i in range(args.calls):
                    call(recs[i % len(recs)], st)
                e1.record(st)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1) / args.calls)
        return ms

    def host_ms(call, kernel_ms):
        call()
        t = []
        for _ in range(5):
            t0 = time.perf_counter()
            call()
            t.append((time.perf_counter() - t0) * 1e3)
        return {"wall_ms_best": min(t), "wall_ms_median": float(np.median(t)), "kernel_ms": kernel_ms()}

    cases = {}

    def case(name, nbytes, dev_call, recs, host_call, kernel_ms, note):
        d = device_ms(dev_call, recs)
        h = host_ms(host_call, kernel_ms)
        best = min(d)
        cases[name] = {"device_ms_per_call": best, "device_ms_windows": d, "host_call": h, "bytes_per_call": int(nbytes),
                       "achieved_gbs": nbytes / (best * 1e-3) / 1e9, "frac_of_copy_peak": nbytes / (best * 1e-3) / 1e9 / HBM_COPY_PEAK_GBS,
                       "device_vs_host_kernel": best / h["kernel_ms"], "host_wall_over_device": h["wall_ms_best"] / best, "note": note}

    # ---- cdfzonal: the inputs of bench.py's siblings()
    msk = m.tmask[:nk].astype(np.float32)
    zm = np.stack([msk[0], m.tmaskatl, np.minimum(1.0, m.tmaskind + m.tmaskpac), m.tmaskind, m.tmaskpac], -1).astype(np.float32)
    e2 = (m.e1v * np.float32(0.75)).astype(np.float32)
    shape = lib.cdfzonal_setup(m.e1v, e2, zm, msk)
    zrec = [synth.make_v_record(m, 3 + r)[:nk].astype(np.float32) for r in range(2)]
    d_z = [dev(z) for z in zrec]
    h_z = pinned(lib, zrec[0], keep)
    o = torch.empty(shape, dtype=torch.float64, device="cuda")
    omx, omn = (torch.empty(shape, dtype=torch.float32, device="cuda") for _ in range(2))
    case("cdfzonal_sum", n3 * 8, lambda z, s: lib.cdfzonal_sum_device(z, o, stream=s), d_z,
         lambda: lib.cdfzonal_sum(h_z, shape), lib.cdfzonal_kernel_ms, "K4, 5 basins; zv + level mask")
    case("cdfzonal_mean", n3 * 8, lambda z, s: lib.cdfzonal_mean_device(z, o, stream=s), d_z,
         lambda: lib.cdfzonal_mean(h_z, shape), lib.cdfzonal_kernel_ms, "K4 mean")
    case("cdfzonal_mean_max", n3 * 8, lambda z, s: lib.cdfzonal_mean_device(z, o, 0.0, True, omx, omn, stream=s), d_z,
         lambda: lib.cdfzonal_mean(h_z, shape, 0.0, True), lib.cdfzonal_kernel_ms, "K4 mean -max (the literal chain)")
    lib.cdfzonal_teardown()
    del d_z

    # ---- cdfmhst
    dims = lib.cdfmhst_setup(m.e1v, m.e3v_0, m.vmask[0].astype(np.float32), m.tmaskatl, m.tmaskpac, m.tmaskind)
    mrec = [((synth.make_v_record(m, 4 + r) * 10.0).astype(np.float32), (synth.make_v_record(m, 6 + r) * 35.0).astype(np.float32))
            for r in range(2)]
    vts = [(synth.make_v_record(m, 8 + r),) + tuple(synth.make_ts_record(m, r)) for r in range(2)]
    d_m = [tuple(dev(a) for a in r) for r in mrec]
    d_v = [tuple(dev(a) for a in r) for r in vts]
    h_m = [pinned(lib, a, keep) for a in mrec[0]]
    h_v = [pinned(lib, a, keep) for a in vts[0]]
    heat, salt = (torch.empty((1, 4, ny), dtype=torch.float64, device="cuda") for _ in range(2))
    case("cdfmhst_vt", n3z * 12, lambda r, s: lib.cdfmhst_record_device(*r, heat, salt, stream=s), d_m,
         lambda: lib.cdfmhst_record(*h_m, dims), lib.cdfmhst_kernel_ms, "K5: vomevt + vomevs + e3v")
    case("cdfmhst_vts", n3z * 32, lambda r, s: lib.cdfmhst_record_vts_device(*r, heat, salt, stream=s), d_v,
         lambda: lib.cdfmhst_record_vts(*h_v, dims), lib.cdfmhst_kernel_ms,
         "K5v (V, T, S read, two products written: 20 B per cell) then K5 (12 B); host kernel_ms is K5 alone")
    lib.cdfmhst_teardown()
    del d_m, d_v

    # ---- cdftransig: one frame, as bench.py's siblings()
    pref, nb, smin, scal, zoom, smn = lib.TRANSIG_CODES["1000"]
    _, _, itab, scm = lib.transig_bins(nb, smin, scal, zoom, smn)
    e2u = (m.e1u * np.float32(0.9)).astype(np.float32)
    e3u = (m.e3v_0 * np.float32(1.01)).astype(np.float32)
    lib.cdftransig_setup(e2u, m.e1v, e3u[:nk], m.e3v_0[:nk], m.nz, nb, pref, smin, scm, itab)
    frames = []
    for r in range(2):
        zt, zs = (x[:nk] for x in synth.make_ts_record(m, r))
        frames.append(((synth.make_v_record(m, 6 + r)[:nk] * m.umask[:nk]).astype(np.float32),
                       (synth.make_v_record(m, 3 + r)[:nk] * m.vmask[:nk]).astype(np.float32), zt, zs))
    d_t = [tuple(dev(a) for a in f) for f in frames]
    h_t = [pinned(lib, a, keep) for a in frames[0]]
    case("cdftransig_frame", n3 * 80, lambda f, s: lib.cdftransig_record_device(*f, False, stream=s), d_t,
         lambda: lib.cdftransig_record(*h_t, False), lib.cdftransig_kernel_ms, "K6, 93 classes; about 80 B per level-cell")
    lib.cdftransig_teardown()
    del d_t

    res = {"tool": "tools/sibling_device_bench.py", **card(), "grid": "ORCA025 L75 (%d x %d x %d)" % (nx, ny, m.nz),
           "calls_per_window": args.calls, "records_in_rotation": 2, "record_mb": n3 * 4 / 1e6, "cases": cases}
    for p in keep:
        p.free()
    lib.finalize()
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).mkdir(parents=True, exist_ok=True)
        (Path(args.out) / "sibling_device.json").write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
