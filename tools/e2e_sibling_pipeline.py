"""The sibling record pipelines against the synchronous calls, ORCA025 L75, records read from files on tmpfs.

    python tools/e2e_sibling_pipeline.py [--out DIR] [--reps N] [--records N]

(a) the C ABI: for cdfzonal (sum), cdfmhst (-v -t -s, _vts) and cdftransig, one loop over the records of float32 (raw
    big-endian, K3 swap) and 16-bit packed (big-endian, K3b unpack) files, each field read with os.preadv straight into a
    pinned buffer; once with the synchronous calls, once with submit / fetch (cdftransig: submit / wait, two slots), the
    two alternating.  Host clock per loop -> ms per record; the results of the two loops are compared bit for bit.  Also the
    H2D ceiling (cdfgpu_h2d_probe) and the read rate of the same preadv calls alone.  With two or more GPUs, the zonal and
    mhst pipelines again under time sharding over all of them.
(b) the command-line twins (cdfzonalsum_gpu, cdfmhst_gpu -v -t -s, cdftransig_xy3d_gpu -S) on the same files: the
    "records" phase of $CDFGPU_TIMING, on one GPU and, when there are several, on all of them.
Prints one JSON line (and writes it to DIR/e2e_sibling_pipeline.json with --out).  Needs a GPU: there is no CPU fallback.
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

from e2e_packed import card                                     # noqa: E402
from e2e_siblings import PACK, SP, records, write_grid          # noqa: E402

GRIDS = {"vozocrtx": ("U", "depthu"), "vomecrty": ("V", "depthv"), "votemper": ("T", "deptht"), "vosaline": ("S", "deptht")}
TOOLS = {"zonal": ("vomecrty",), "mhst": ("vomecrty", "votemper", "vosaline"), "transig": ("vozocrtx", "vomecrty", "votemper", "vosaline")}


class Field:
    """The field of a file of write_grid: two record variables, time_counter (8 bytes) then the field, so record r of the
    field is the byte range begin + r * (8 + vsize) (vsize is a multiple of 4: no padding)."""

    def __init__(self, path, name, nrec, n3, esize):
        from scipy.io import netcdf_file
        self.fd = os.open(path, os.O_RDONLY)
        self.vsize = n3 * esize
        self.recsize = 8 + self.vsize
        self.begin = os.fstat(self.fd).st_size - nrec * self.recsize + 8
        f = netcdf_file(str(path), "r", mmap=False)   # the layout is checked on the last values of the last record
        want = np.ascontiguousarray(f.variables[name][nrec - 1].ravel()[-64:]).astype(">f4" if esize == 4 else ">i2").tobytes()
        f.close()
        assert os.pread(self.fd, 64 * esize, self.begin + (nrec - 1) * self.recsize + self.vsize - 64 * esize) == want, path

    def read(self, r, pinned):
        mv = memoryview(pinned.array.view(np.uint8).reshape(-1))[:self.vsize]
        assert os.preadv(self.fd, [mv], self.begin + r * self.recsize) == self.vsize


def abi(lib, m, d, nrec, reps, ndev):
    import oracle
    nz, ny, nx = m.e3v_0.shape
    n3 = nz * ny * nx
    msk = m.vmask.astype(np.float32)
    out = {}
    for kind in ("float", "packed"):
        esize = 4 if kind == "float" else 2
        fields = {f: Field(d / kind / f"grid{GRIDS[f][0]}.nc", f, nrec, n3, esize) for f in GRIDS}
        ns = lib.nslots()
        bufs = [{f: lib.PinnedArray((n3,), np.float32 if esize == 4 else np.int16) for f in GRIDS} for _ in range(max(ns, 2))]
        for call, names in ((lib.CALL_ZONAL, ("vomecrty",)), (lib.CALL_MHST_VTS, TOOLS["mhst"]), (lib.CALL_TRANSIG, TOOLS["transig"])):
            for fi, f in enumerate(names):
                if kind == "packed":
                    lib.set_sibling_input(call, fi, lib.INPUT_I16, True, *PACK[f], SP)
                else:
                    lib.set_sibling_input(call, fi, lib.INPUT_F32, True)
        zshape = lib.cdfzonal_setup(m.e1v, m.e1v, oracle.zonal_masks(msk[0], m.tmaskatl, m.tmaskind, m.tmaskpac), msk)
        mdims = lib.cdfmhst_setup(m.e1v, m.e3v_0, msk[0], m.tmaskatl, m.tmaskpac, m.tmaskind)
        pref, nb, smin, scal, zoom, smn = lib.TRANSIG_CODES["1000"]
        _, _, itab, step = lib.transig_bins(nb, smin, scal, zoom, smn)
        tsetup = lambda: lib.cdftransig_setup(m.e1u, m.e1v, m.e3v_0[:-1], m.e3v_0[:-1], nz, nb, pref, smin, step, itab, lperio=True)

        def read(tool, r, b):
            for f in TOOLS[tool]:
                fields[f].read(r, b[f])

        def sync(tool):
            res = []
            if tool == "transig":
                tsetup()
            for r in range(nrec):
                b = bufs[0]
                read(tool, r, b)
                if tool == "zonal":
                    res.append(lib.cdfzonal_sum(b["vomecrty"].array, zshape))
                elif tool == "mhst":
                    res.append(lib.cdfmhst_record_vts(*(b[f].array for f in TOOLS["mhst"]), mdims))
                else:
                    lib.cdftransig_record(*(b[f].array for f in TOOLS["transig"]), set_masks=r < nrec // 2)
            return res if tool != "transig" else list(lib.cdftransig_fetch((nb, ny, nx)))

        def piped(tool):
            res = [None] * nrec
            nsl = 2 if tool == "transig" else ns
            if tool == "transig":
                tsetup()
            fetch = (lambda s: lib.cdfzonal_fetch(s, zshape)) if tool == "zonal" else (lambda s: lib.cdfmhst_fetch(s, mdims))
            for r in range(nrec):
                s = r % nsl
                if r >= nsl:
                    if tool == "transig":
                        lib.cdftransig_wait(s)
                    else:
                        res[r - nsl] = fetch(s)
                b = bufs[s]
                read(tool, r, b)
                if tool == "zonal":
                    lib.cdfzonal_submit_sum(s, b["vomecrty"].array)
                elif tool == "mhst":
                    lib.cdfmhst_submit_vts(s, *(b[f].array for f in TOOLS["mhst"]))
                else:
                    lib.cdftransig_submit(s, *(b[f].array for f in TOOLS["transig"]), set_masks=r < nrec // 2)
            if tool == "transig":
                return list(lib.cdftransig_fetch((nb, ny, nx)))
            for r in range(max(0, nrec - nsl), nrec):
                res[r] = fetch(r % nsl)
            return res

        def flat(x):
            return [a for y in x for a in (y if isinstance(y, tuple) else (y,))]

        res = {}
        for tool in TOOLS if ndev == 1 else ("zonal", "mhst"):
            sync(tool), piped(tool)   # warm-up: staging buffers, slot buffers
            t = {"sync": [], "pipeline": []}
            outs = {}
            for _ in range(reps):
                for way, fn in (("sync", sync), ("pipeline", piped)):
                    t0 = time.perf_counter()
                    outs[way] = fn(tool)
                    t[way].append((time.perf_counter() - t0) / nrec * 1e3)
            nbytes = n3 * esize * len(TOOLS[tool])
            res[tool] = {w: {"ms_per_record": float(np.median(v)), "ms_min": min(v), "ms_max": max(v), "ms_all": v} for w, v in t.items()}
            res[tool]["h2d_bytes_per_record"] = nbytes
            res[tool]["speedup"] = res[tool]["sync"]["ms_per_record"] / res[tool]["pipeline"]["ms_per_record"]
            res[tool]["results_identical"] = all(np.array_equal(a, b, equal_nan=True) for a, b in zip(flat(outs["sync"]), flat(outs["pipeline"])))
            # read alone: the same preadv calls of all records
            t0 = time.perf_counter()
            for r in range(nrec):
                read(tool, r, bufs[0])
            dt = time.perf_counter() - t0
            res[tool]["read_ms_per_record"] = dt / nrec * 1e3
            res[tool]["read_gbs"] = nbytes * nrec / dt / 1e9
        res["h2d_ceiling_gbs"] = lib.h2d_probe(bufs[0]["vomecrty"], reps=6)
        out[kind] = res
        lib.cdfzonal_teardown()
        lib.cdfmhst_teardown()
        for b in bufs:
            for p in b.values():
                p.free()
        for f in fields.values():
            os.close(f.fd)
    return out


def twins(d, ndevs):
    from cdftools_b200 import build
    cases = {"cdfzonalsum_gpu": ["-f", "gridV.nc", "-p", "V"], "cdfmhst_gpu": ["-v", "gridV.nc", "-t", "gridT.nc", "-s", "gridS.nc"],
             "cdftransig_xy3d_gpu": ["-c", "SYN", "-l", "y2026", "-S"]}
    outs = {"cdfzonalsum_gpu": ["zonalsum.nc"], "cdfmhst_gpu": ["mhst.nc", "zonal_heat_trp.dat"], "cdftransig_xy3d_gpu": ["uvxysig.nc"]}
    res, files = {}, {}
    with tempfile.TemporaryDirectory() as bindir:
        tools = build.build_host(bindir=bindir, names=list(cases))
        for n in ndevs:
            env = dict(os.environ, CDFGPU_TIMING="1", CDFGPU_DEVICES=str(n), CDFGPU_SHARD="time")
            rec = {t: {"float": [], "packed": []} for t in cases}
            for it in range(3):
                for tool, args in cases.items():
                    for kind in ("float", "packed"):
                        r = subprocess.run([str(tools[tool])] + args, cwd=d / kind, check=True, capture_output=True, text=True, env=env)
                        ph = {l.split()[2]: float(l.split()[3]) for l in r.stderr.splitlines() if l.startswith(tool + ": phase")}
                        if it:   # the first round warms the page cache
                            rec[tool][kind].append(ph["records"])
                        files[n, tool, kind] = [(d / kind / o).read_bytes() for o in outs[tool]]
            res["gpus_%d" % n] = {"records_phase_s": {t: {k: min(v) for k, v in r.items()} for t, r in rec.items()},
                                  "records_phase_s_all": rec}
        res["float_and_packed_outputs_identical"] = {t: files[1, t, "float"] == files[1, t, "packed"] for t in cases}
        if len(ndevs) > 1:
            res["outputs_identical_across_gpu_counts"] = {t: all(files[n, t, k] == files[1, t, k] for n in ndevs for k in ("float", "packed"))
                                                         for t in cases}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--records", type=int, default=8)
    a = ap.parse_args()
    from cdftools_b200 import lib, ncfiles, synth
    res = {"tool": "tools/e2e_sibling_pipeline.py", **card()}
    m = synth.make_mesh("ORCA025")
    res["grid"] = "ORCA025 L75 (%d x %d x %d)" % (m.nx, m.ny, m.nz)
    res["records_per_file"] = a.records
    ngpu = lib.device_count()
    with tempfile.TemporaryDirectory(dir="/dev/shm" if Path("/dev/shm").exists() else None) as d:
        d = Path(d)
        ncfiles.write_mesh(m, d / "mesh")
        recs = [records(m, r) for r in range(a.records)]
        for kind in ("float", "packed"):
            (d / kind).mkdir()
            for mf in (d / "mesh").iterdir():
                (d / kind / mf.name).symlink_to(mf)
            for name, (g, zdim) in GRIDS.items():
                write_grid(d / kind / f"grid{g}.nc", m, zdim, name, [r[name] for r in recs], kind == "packed")
                (d / kind / f"SYN_y2026_grid{g}.nc").symlink_to(d / kind / f"grid{g}.nc")
        del recs
        lib.init(0, 3)
        try:
            res["abi_1gpu"] = abi(lib, m, d, a.records, a.reps, 1)
        finally:
            lib.finalize()
        if ngpu >= 2:
            lib.init_multi(min(ngpu, 8), "time", 3)
            try:
                res["abi_%dgpu_time_sharded" % min(ngpu, 8)] = abi(lib, m, d, a.records, a.reps, min(ngpu, 8))
            finally:
                lib.finalize()
        res["twins"] = twins(d, [1] + ([min(ngpu, 8)] if ngpu >= 2 else []))
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).mkdir(parents=True, exist_ok=True)
        (Path(a.out) / "e2e_sibling_pipeline.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
