"""cdfsigtrp on a device-resident record (cdfsigtrp_gpu_sections_setup / _device) against the host path it replaces,
ORCA025 L75, one process on one GPU.

    python tools/sigtrp_device_bench.py [--out DIR] [--calls N]

Setup: one synthetic ORCA025 L75 record of U, V, T, S resident on the GPU; 30 sections, zonal and meridional in turn, of 2
to 1400 columns (geometric spread, the meridional ones capped at 1000); sigma0, 100 classes.
  * device path: N calls (after a warm-up) on a torch stream, timed with CUDA events on that stream; per call = window / N,
    three windows.  Launches per call from cdfgpu_launch_count.  The kernel time per call is read from a torch.profiler
    trace of 20 further calls (a run of its own): when the window is no longer than the kernels, the event time is GPU
    time; when it is longer, the host's enqueue rate sets it.
  * host path: what a caller without the batched call does for the same sections -- cut the slices out of the host record
    with numpy, prepare them as src/cdfsigtrp.f90:428-555 (the C reference implementation), and one cdfsigtrp_gpu_section
    per section; host clock around the whole list (best and median of 5).
  * whether every section's binned transports and nk are bit-identical on the two paths.
The GPU's name and power limit are read in the same run.  Prints one JSON line (and writes DIR/sigtrp_device.json with
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


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or ["?, ?"])[0].split(",", 1)
    return {"gpu": name.strip(), "power_limit": power.strip()}


def section_boxes(nx, ny, n=30):
    """n sections, zonal and meridional in turn, 2 .. 1400 columns, spread over the grid."""
    lengths = np.unique(np.round(np.geomspace(2, 1400, n)).astype(int))
    while lengths.size < n:
        lengths = np.unique(np.append(lengths, lengths[-1] - lengths.size))
    boxes = []
    for s, npts in enumerate(sorted(lengths)):
        if s % 2 == 1:   # zonal (the longest one too), rows spread from south to north
            npts = min(int(npts), nx - 2)
            j = 40 + (s * 37) % (ny - 80)
            i0 = 1 + (s * 53) % (nx - npts - 1)
            boxes.append((i0, i0 + npts, j, j))
        else:
            npts = min(int(npts), 1000)
            i = 1 + (s * 97) % (nx - 2)
            j0 = (s * 29) % (ny - npts - 1)
            boxes.append((i, i, j0, j0 + npts))
    return boxes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--calls", type=int, default=200)
    args = ap.parse_args()
    import torch
    import oracle
    from cdftools_b200 import lib, ncfiles, synth

    oracle.build()
    lib.init(0, 3)
    m = synth.make_mesh("ORCA025")
    nx, ny, npk = m.nx, m.ny, m.nz
    f32 = np.float32
    u = (synth.make_v_record(m, 500) * m.umask).astype(f32)
    v = synth.make_v_record(m, 0)
    t, s = synth.make_ts_record(m, 0)
    e3w_1d, e3w = ncfiles.e3w_fields(m)
    e2u, e3u = (m.e1u * f32(0.9)).astype(f32), (m.e3v_0 * f32(1.01)).astype(f32)
    boxes = section_boxes(nx, ny)
    mode, refdep, smin, smax, nbins = 0, 0.0, 23.0, 28.5, 100
    nsec = len(boxes)

    t0 = time.perf_counter()
    lev, npts = lib.cdfsigtrp_sections_setup(np.array(boxes), m.gdept_1d, m.gdepw_1d, smin, smax, nbins, e1v=m.e1v, e2u=e2u, e3u=e3u,
                                             e3v=m.e3v_0, e3w=e3w, mode=mode, refdep=refdep)
    setup_ms = (time.perf_counter() - t0) * 1e3
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    d = [dev(a) for a in (u, v, t, s)]
    out = torch.empty((nsec, nbins), dtype=torch.float64, device="cuda")
    d_nk = torch.empty(nsec, dtype=torch.int32, device="cuda")
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(st):
        for _ in range(10):
            lib.cdfsigtrp_sections_device(*d, out, d_nk, stream=st)
    torch.cuda.synchronize()
    n0 = lib.launch_count()
    windows = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(st):
            e0.record(st)
            for _ in range(args.calls):
                lib.cdfsigtrp_sections_device(*d, out, d_nk, stream=st)
            e1.record(st)
        e1.synchronize()
        windows.append(e0.elapsed_time(e1) / args.calls)
    launches = (lib.launch_count() - n0) / (3 * args.calls)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        with torch.cuda.stream(st):
            for _ in range(20):
                lib.cdfsigtrp_sections_device(*d, out, d_nk, stream=st)
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.events():
        if "sigtrp_sections_" in e.name and e.device_time > 0:   # microseconds
            k = e.name.split("sigtrp_sections_")[1].split("_kernel")[0]
            kernels[k] = kernels.get(k, 0.0) + e.device_time / 20 / 1e3
    kernel_ms = sum(kernels.values())
    got, got_nk = out.cpu().numpy(), d_nk.cpu().numpy()

    def host_path():
        rows, nks = [], []
        for sec in boxes:
            imin, imax, jmin, jmax = sec
            if imin == imax:
                r, i0 = slice(jmin, jmax), imin - 1
                c = lambda a, i: np.ascontiguousarray(a[:, r, i])
                eu, de3, zu, a, b = e2u[r, i0].copy(), c(e3u, i0), c(u, i0), i0, i0 + 1
            else:
                cols, j0 = slice(imin, imax), jmin - 1
                c = lambda a, j: np.ascontiguousarray(a[:, j, cols])
                eu, de3, zu, a, b = m.e1v[j0, imin - 1:imax - 1].copy(), c(m.e3v_0, j0), c(v, j0), j0, j0 + 1
            p = oracle.sigtrp_prepare(m.gdept_1d[0], c(e3w, a), c(e3w, b), zu, 0.0, c(s, a), c(s, b), 0.0, c(t, a), c(t, b),
                                      merid=imin == imax)
            o = lib.cdfsigtrp_section(eu, de3, p["ddepu"], m.gdepw_1d, p["zu"], p["zt"], p["zs"], p["zmask"], p["nk"], smin, smax,
                                      nbins, mode=mode, refdep=refdep)
            rows.append(o["dtrpbin"])
            nks.append(p["nk"])
        return np.array(rows), np.array(nks)

    ref, ref_nk = host_path()
    wall = []
    for _ in range(5):
        t0 = time.perf_counter()
        host_path()
        wall.append((time.perf_counter() - t0) * 1e3)
    best = min(windows)
    res = {"tool": "tools/sigtrp_device_bench.py", **card(), "grid": "ORCA025 L75 (%d x %d x %d)" % (nx, ny, npk),
           "sections": nsec, "columns": int(npts.sum()), "npts_min": int(npts.min()), "npts_max": int(npts.max()),
           "zonal": sum(1 for b in boxes if b[0] != b[1]), "meridional": sum(1 for b in boxes if b[0] == b[1]),
           "classes": nbins, "mode": "sigma0", "calls_per_window": args.calls,
           "device_ms_per_call": best, "device_ms_windows": windows, "launches_per_call": launches,
           "kernel_ms_per_call_trace": kernel_ms, "kernel_ms_by_kernel_trace": kernels, "device_over_kernel": best / kernel_ms,
           "setup_ms_host_clock": setup_ms,
           "host_path_ms_best": min(wall), "host_path_ms_median": float(np.median(wall)),
           "host_path_launches_per_call": 4 * nsec, "host_over_device": min(wall) / best,
           "bit_identical_dtrpbin": bool(np.array_equal(got, ref, equal_nan=True)),
           "bit_identical_nk": bool(np.array_equal(got_nk, ref_nk)), "nonzero_bins": int(np.count_nonzero(got)),
           "boxes": [list(map(int, b)) for b in boxes]}
    lib.finalize()
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).mkdir(parents=True, exist_ok=True)
        (Path(args.out) / "sigtrp_device.json").write_text(json.dumps(res, indent=1) + "\n")
    if not (res["bit_identical_dtrpbin"] and res["bit_identical_nk"]):
        sys.exit("the two paths differ")


if __name__ == "__main__":
    main()
