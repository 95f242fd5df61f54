"""Latitude-band sharding of the sibling tools (CDFGPU_SHARD=lat) on 1, 2, 4, 8 devices, ORCA025 L75, one process.

    python tools/sibling_bands_bench.py [--out DIR] [--ndev 1,2,4,8] [--frames 8] [--records 16] [--orca12]

Loops, each on seeded synthetic records (cdftools_b200.synth) in pinned host buffers (a record is ~440 MB, far above the
126 MB L2), for every N the box has:
  * cdftransig frame pipeline: -code 1000 (93 bins), fixed e3, `--frames` frames through 3 slots (wait before a slot is
    reused), timed up to the end of the last frame's kernels; the fetch of the sums (2 x 1.1 GB into pageable host arrays)
    is timed on its own;
  * cdfmhst_gpu_submit_vts and cdfzonal_gpu_submit_sum pipelines: `--records` records through the slots, each fetched
    before its slot is reused; beside them the time-sharded figure at the same N (3 slots per device).
Per run: wall time per record (host clock around the loop, which ends in a blocking fetch or wait; best of two passes after
a warm-up pass), bytes copied host -> device per record (halo rows included) and GB/s, device memory each device holds after
the run (cudaMemGetInfo before setup and before teardown), and whether the results equal those of N = 1 bit for bit.
--orca12: one more cdftransig run at ORCA12 width with -code 2000 (174 bins), when the host has the memory for it.
The GPUs' name and power limit are read in the same run.  Prints one JSON line, and writes DIR/r07_sibling_bands.json with
--out.  Needs GPUs: there is no CPU fallback.
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
    rows = [l.split(",", 1) for l in r.stdout.strip().splitlines() if "," in l]
    return {"gpu": rows[0][0].strip() if rows else "?", "power_limit": sorted({p.strip() for _, p in rows}) or ["?"]}


def host_gb_available():
    for line in Path("/proc/meminfo").read_text().splitlines():
        if line.startswith("MemAvailable:"):
            return int(line.split()[1]) / 1e6
    return 0.0


def pinned(lib, a, keep):
    p = lib.PinnedArray(a.shape, a.dtype)
    p.array[...] = a
    keep.append(p)
    return p.array


def band_rows(ny, n, halo):
    """rows each device holds under latitude sharding (the plan of libcdfgpu: nb = min(n, ny) balanced bands)"""
    from cdftools_b200.shard import band_plan
    b = band_plan(ny, min(n, ny))
    return [j1 - j0 + (halo if d < len(b) - 1 else 0) for d, (j0, j1) in enumerate(b)]


class Session:
    def __init__(self, lib, torch, n, shard):
        self.lib, self.torch, self.n = lib, torch, n
        lib.finalize()
        if n == 1:
            lib.init(0, 3)
        else:
            lib.init_multi(n, shard, 3)
        self.free0 = self.free()

    def free(self):
        return [self.torch.cuda.mem_get_info(d)[0] for d in range(self.n)]

    def held_gb(self):
        return [round((a - b) / 1e9, 3) for a, b in zip(self.free0, self.free())]


def timed(run, passes=3):
    """best wall time (s) of passes 2..: the first one warms up"""
    best, out = None, None
    for p in range(passes):
        t0 = time.perf_counter()
        out = run()
        dt = time.perf_counter() - t0
        if p > 0:
            best = dt if best is None else min(best, dt)
    return best, out


def pipeline(lib, n, submit, fetch):
    ns = lib.nslots()
    out = [None] * n
    for r in range(n):
        if r >= ns:
            out[r - ns] = fetch((r - ns) % ns)
        submit(r % ns, r)
    for r in range(max(0, n - ns), n):
        out[r] = fetch(r % ns)
    return out


def transig_run(lib, torch, n, m, frames, code, nframes):
    pref, nb, smin, scal, zoom, smn = lib.TRANSIG_CODES[code]
    _, _, itab, step = lib.transig_bins(nb, smin, scal, zoom, smn)
    e2u = (m.e1u * np.float32(0.9)).astype(np.float32)
    e3u = (m.e3v_0[:-1] * np.float32(1.01)).astype(np.float32)
    s = Session(lib, torch, n, "lat")

    def run():
        shape = lib.cdftransig_setup(e2u, m.e1v, e3u, m.e3v_0[:-1], m.nz, nb, pref, smin, step, itab)   # zeroes the sums
        t0 = time.perf_counter()
        for r in range(nframes):
            if r >= 3:
                lib.cdftransig_wait(r % 3)
            lib.cdftransig_submit(r % 3, *frames[r % len(frames)], set_masks=r < nframes // 2)
        lib.cdftransig_kernel_ms()   # blocks until the last frame's kernels are done
        t1 = time.perf_counter()
        out = lib.cdftransig_fetch(shape)
        return t1 - t0, time.perf_counter() - t1, out

    runs = [run() for _ in range(3)]   # the first one warms up
    frames_s = min(r[0] for r in runs[1:])
    fetch_s = min(r[1] for r in runs[1:])
    held = s.held_gb()
    lib.cdftransig_teardown()
    copied = sum(band_rows(m.ny, n, 1)) * m.nx * (m.nz - 1) * 4 * 4
    return {"ms_per_frame": round(frames_s / nframes * 1e3, 3), "bytes_per_frame": copied,
            "gbs": round(copied / (frames_s / nframes) / 1e9, 2), "fetch_ms": round(fetch_s * 1e3, 1),
            "device_mem_gb": held}, runs[-1][2]


def sibling_run(lib, torch, n, shard, setup, submit, fetch, nrec, bytes_per_device_rec):
    s = Session(lib, torch, n, shard)
    teardown = setup()
    best, out = timed(lambda: pipeline(lib, nrec, submit, fetch))
    held = s.held_gb()
    teardown()
    return {"ms_per_record": round(best / nrec * 1e3, 3), "bytes_per_record": bytes_per_device_rec,
            "gbs": round(bytes_per_device_rec / (best / nrec) / 1e9, 2), "device_mem_gb": held}, out


def equal(a, b):
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(equal(x, y) for x, y in zip(a, b))
    return bool(np.array_equal(a, b, equal_nan=True))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--ndev", default="1,2,4,8")
    ap.add_argument("--frames", type=int, default=8)
    ap.add_argument("--records", type=int, default=16)
    ap.add_argument("--orca12", action="store_true")
    args = ap.parse_args()
    import torch
    from cdftools_b200 import lib, synth

    lib.init(0, 3)
    ndevs = [n for n in (int(x) for x in args.ndev.split(",")) if n <= lib.device_count()]
    res = {"what": "sibling tools under CDFGPU_SHARD=lat, ORCA025 L75, one process", **card(), "devices": lib.device_count(),
           "transig": {}, "mhst_vts": {}, "zonal_sum": {}}
    m = synth.make_mesh("ORCA025")
    nx, ny, nz = m.nx, m.ny, m.nz
    keep = []
    # cdftransig: two frames in rotation (zu, zv, zt, zs levels 1..nz-1)
    frames = []
    for r in range(2):
        t, s = synth.make_ts_record(m, r)
        frames.append([pinned(lib, np.ascontiguousarray(a[:-1]), keep)
                       for a in ((synth.make_v_record(m, 500 + r) * m.umask), synth.make_v_record(m, r), t, s)])
    ref = None
    for n in ndevs:
        r, out = transig_run(lib, torch, n, m, frames, "1000", args.frames)
        ref = out if ref is None else ref
        r["bit_identical_to_n1"] = equal(out, ref)
        res["transig"][str(n)] = r
        print(json.dumps({"transig": n, **r}), file=sys.stderr, flush=True)
    for p in keep:
        p.free()
    keep.clear()
    # cdfmhst -v/-t/-s and cdfzonalsum: three records in rotation
    recs = []
    for r in range(3):
        t, s = synth.make_ts_record(m, r)
        recs.append([pinned(lib, np.ascontiguousarray(a), keep) for a in (synth.make_v_record(m, r), t, s)])
    e2 = (m.e1v * np.float32(0.75)).astype(np.float32)
    msk = m.vmask[:-1].astype(np.float32)
    import oracle
    zm = oracle.zonal_masks(msk[0], m.tmaskatl, m.tmaskind, m.tmaskpac)
    alpha = (0.5 + np.arange(ny) / ny).astype(np.float32)
    dims, zshape = (nz, ny), None

    def mhst_setup():
        lib.cdfmhst_setup(m.e1v, m.e3v_0, m.vmask[0].astype(np.float32), m.tmaskatl, m.tmaskpac, m.tmaskind)
        return lib.cdfmhst_teardown

    def zonal_setup():
        nonlocal zshape
        zshape = lib.cdfzonal_setup(m.e1v, e2, zm, msk)
        return lib.cdfzonal_teardown

    refs = {}
    for n in ndevs:
        for shard in (("lat", "time") if n > 1 else ("lat",)):
            key = str(n) if shard == "lat" else f"{n}_time"
            halo_rows = sum(band_rows(ny, n, 1)) if shard == "lat" else ny
            r, out = sibling_run(lib, torch, n, shard, mhst_setup, lambda sl, i: lib.cdfmhst_submit_vts(sl, *recs[i % 3]),
                                 lambda sl: lib.cdfmhst_fetch(sl, dims), args.records, 3 * nz * halo_rows * nx * 4)
            refs.setdefault("mhst", out)
            r["bit_identical_to_n1"] = equal(out, refs["mhst"])
            res["mhst_vts"][key] = r
            print(json.dumps({"mhst_vts": key, **r}), file=sys.stderr, flush=True)
            r, out = sibling_run(lib, torch, n, shard, zonal_setup, lambda sl, i: lib.cdfzonal_submit_sum(sl, recs[i % 3][0][:-1], alpha),
                                 lambda sl: lib.cdfzonal_fetch(sl, zshape), args.records, (nz - 1) * ny * nx * 4)
            refs.setdefault("zonal", out)
            r["bit_identical_to_n1"] = equal(out, refs["zonal"])
            res["zonal_sum"][key] = r
            print(json.dumps({"zonal_sum": key, **r}), file=sys.stderr, flush=True)
    for p in keep:
        p.free()
    keep.clear()
    if args.orca12:
        m12 = synth.make_mesh("ORCA12")
        need = 6 * (m12.nz - 1) * m12.ny * m12.nx * 4 / 1e9 * 1.3
        if host_gb_available() < need:
            res["transig_orca12"] = f"not measured: needs ~{need:.0f} GB of host memory"
        else:
            t, s = synth.make_ts_record(m12, 0)
            fr = [pinned(lib, np.ascontiguousarray(a[:-1]), keep)
                  for a in ((synth.make_v_record(m12, 500) * m12.umask), synth.make_v_record(m12, 0), t, s)]
            del t, s
            res["transig_orca12"] = {}
            for n in ndevs:
                if n == 1:
                    continue   # 2 x 174 x 13.2 M x 8 B of accumulators and the frame slots: one device does not hold them
                r, _ = transig_run(lib, torch, n, m12, [fr], "2000", 4)
                res["transig_orca12"][str(n)] = r
                print(json.dumps({"transig_orca12": n, **r}), file=sys.stderr, flush=True)
            for p in keep:
                p.free()
    lib.finalize()
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).mkdir(parents=True, exist_ok=True)
        (Path(args.out) / "r07_sibling_bands.json").write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
