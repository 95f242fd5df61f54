"""K1 (moc_zonal_scan_kernel) on the bench's ORCA025 L75 case: time per record and achieved bandwidth on the bytes the kernel
has to move now that it skips the zero area vectors, one process on one GPU.  CDFGPU_LIB selects another build of the
library (tools/ab_variants.sh), for A/B runs in one process per library.

    python tools/k1_zero_area_bench.py [--out DIR] [--records N] [--reps R]

Setup as bench.py builds it: synth.make_mesh("ORCA025"), setup_masks, setup_e3v_masked; N distinct V records of
randn * 0.1 * vmask resident on the GPU (73 by default: 31.8 GB, far larger than the 126 MB L2).
  * bytes, counted on the host from the same mesh: area = fl32(e1v * e3m) over levels 0..nz-2 as the setup kernel forms it,
    the fraction f of flat 16-byte area vectors with a non-zero word, and per record
      needed      = V (4 B per level-cell) + 16 B per non-zero area vector + mask bytes (ny*nx) + output (nb*ny*nz*8)
      algorithmic = V + the whole area field (8 B per level-cell) + mask + output, what bench.py's roofline counts;
  * time: CUDA events on one stream around R passes over the N records, batched (cdfmoc_gpu_compute_device_batch, one launch
    per pass) and one launch per record (cdfmoc_gpu_compute_device, what the submit pipeline issues), after one warm-up pass;
    best and median of the R passes;
  * the device-to-device copy bandwidth of this GPU, measured in the same run (torch copy of 4 GiB, read + write bytes);
  * the GPU's name, power limit and maximum SM clock (nvidia-smi, query only);
  * K1's basin words on the same mesh, counted on the host as pack_masks (api.cu) builds them: the in-row cells with a
    non-zero basin byte that carry their vector's lead byte, and the others (exceptions) per (j,k) row, which K1 adds cell
    by cell.
Prints one JSON line (and writes DIR/k1_zero_area.json with --out).  Needs a GPU: there is no CPU fallback.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    f = [x.strip() for x in (r.stdout.strip().splitlines() or ["?, ?, ?"])[0].split(",")]
    return {"gpu": f[0], "power_limit": f[1] if len(f) > 1 else "?", "clocks_max_sm": f[2] if len(f) > 2 else "?"}


def area_bytes(m, e3m):
    """-> (level-cells, non-zero 16-byte area vectors, all vectors) of the resident area field, levels 0..nz-2."""
    area = (m.e1v[None, :, :] * e3m[: m.nz - 1]).astype(np.float32).ravel()
    n = area.size
    w = np.zeros((n + 3) // 4 * 4, np.uint32)
    w[:n] = area.view(np.uint32)
    nz = int(np.count_nonzero(w.reshape(-1, 4).any(axis=1)))
    return n, nz, w.size // 4


def vector_basin_counts(ib, nz):
    """K1's per-vector basin words (pack_masks in api.cu) over the (j,k) rows of one record: the in-row cells with a non-zero
    byte that carry their vector's lead byte, and the others (exceptions) per row, which K1 adds cell by cell, one lane
    each (a row with more than 32 takes the literal chain)."""
    ny, nx, nb = ib.shape
    byt = (ib.astype(np.int32) << np.arange(nb)).sum(axis=2)
    exc_rows, kept, nonzero = [], 0, 0
    for s in range(4):
        w = (s + nx + 3) // 4
        cells = np.full((ny, 4 * w), -1, np.int32)
        cells[:, s:s + nx] = byt
        v = cells.reshape(ny, w, 4)
        n = np.where(v > 0, (v[..., :, None] == v[..., None, :]).sum(axis=-1), 0)
        lead = np.take_along_axis(v, n.argmax(axis=-1)[..., None], axis=-1)   # argmax: ties go to the first cell
        # rows (k, j) whose first cell sits s cells into its vector, k = 0..nz-2
        k = np.arange(nz - 1)[:, None]
        nrows = (((k * ny + np.arange(ny)[None, :]) * nx) % 4 == s).sum(axis=0)
        kept += int((((v > 0) & (v == lead)).sum(axis=(1, 2)) * nrows).sum())
        nonzero += int(((v > 0).sum(axis=(1, 2)) * nrows).sum())
        exc_rows.append(np.repeat(((v > 0) & (v != lead)).sum(axis=(1, 2)), nrows))
    e = np.concatenate(exc_rows)
    return {"mask_bytes_distinct": sorted(int(x) for x in np.unique(byt)), "inrow_nonzero_cells": nonzero,
            "frac_lead_byte": kept / nonzero, "exceptions_per_row_mean": float(e.mean()), "exceptions_per_row_max": int(e.max()),
            "rows_with_exceptions": int((e > 0).sum()), "rows_over_32_exceptions": int((e > 32).sum()), "rows": int(e.size)}


def copy_peak_gbs(torch, nbytes=4 << 30, reps=10):
    a = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    gbs = 2 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del a, b
    torch.cuda.empty_cache()
    return gbs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", type=Path, default=None)
    ap.add_argument("--records", type=int, default=73)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()

    import torch
    from cdftools_b200 import lib, synth
    if not torch.cuda.is_available():
        raise SystemExit("k1_zero_area_bench: no CUDA device -- libcdfgpu has no CPU fallback")

    m = synth.make_mesh("ORCA025")
    ib = synth.setup_masks(m)
    e3m = synth.setup_e3v_masked(m)
    nx, ny, nz, nb = m.nx, m.ny, m.nz, ib.shape[2]
    ncell, nzvec, nvec = area_bytes(m, e3m)
    small = ny * nx + nb * ny * nz * 8
    needed = ncell * 4 + nzvec * 16 + small
    algorithmic = ncell * 8 + small

    peak = copy_peak_gbs(torch)
    lib.init(0, 3)
    lib.set_device_inputs_ready(True)
    try:
        lib.cdfmoc_setup(m.e1v, e3m, ib)
        gen = torch.Generator(device="cuda")
        gen.manual_seed(20261017)
        vmask = torch.from_numpy(m.vmask[:-1].astype(np.float32)).cuda()
        recs = [torch.randn((nz - 1, ny, nx), device="cuda", generator=gen).mul_(0.1).mul_(vmask) for _ in range(args.records)]
        outs = [torch.zeros((nz, ny, nb), dtype=torch.float64, device="cuda") for _ in range(args.records)]
        st = torch.cuda.Stream()

        def timed(batch):
            ms = []
            for rep in range(args.reps + 1):   # the first pass warms up
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                with torch.cuda.stream(st):
                    e0.record(st)
                    if batch:
                        lib.cdfmoc_compute_device_batch(recs, outs, st)
                    else:
                        for r, o in zip(recs, outs):
                            lib.cdfmoc_compute_device(r, o, st)
                    e1.record(st)
                st.synchronize()
                if rep:
                    ms.append(e0.elapsed_time(e1) / args.records)
            best, med = min(ms), float(np.median(ms))
            return {"ms_per_record_best": best, "ms_per_record_median": med,
                    "gbs_needed_bytes": needed / (med * 1e-3) / 1e9, "frac_of_copy_peak_needed_bytes": needed / (med * 1e-3) / 1e9 / peak,
                    "gbs_algorithmic_bytes": algorithmic / (med * 1e-3) / 1e9,
                    "frac_of_copy_peak_algorithmic_bytes": algorithmic / (med * 1e-3) / 1e9 / peak}

        res = {"batched": timed(True), "per_record_launches": timed(False)}
        lib.cdfmoc_teardown()
    finally:
        lib.finalize()

    line = {"tool": "k1_zero_area_bench", "lib": str(lib.SO_PATH.relative_to(ROOT)) if lib.SO_PATH.is_relative_to(ROOT) else str(lib.SO_PATH),
            "grid": "ORCA025", "nx": nx, "ny": ny, "nz": nz, "basins": nb, "records": args.records,
            "reps": args.reps, **card(), "copy_peak_gbs": peak,
            "area_vectors": nvec, "area_vectors_nonzero": nzvec, "f_nonzero": nzvec / nvec,
            "bytes_per_level_cell_needed": 4 + 4 * nzvec / nvec,
            "bytes_per_record_needed": needed, "bytes_per_record_algorithmic": algorithmic,
            "vector_basins": vector_basin_counts(ib, nz), **res,
            "note": "needed = V + non-zero area vectors + masks + output; algorithmic = V + whole area + masks + output "
                    "(bench.py's roofline); copy peak = torch device-to-device copy, read + write bytes, same run"}
    print(json.dumps(line))
    if args.out:
        args.out.mkdir(parents=True, exist_ok=True)
        (args.out / "k1_zero_area.json").write_text(json.dumps(line, indent=2) + "\n")


if __name__ == "__main__":
    main()
