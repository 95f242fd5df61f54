"""16-bit packed records on the device (K3b) against float32 records, ORCA025 L75 cdfmoc, in one process on one GPU.

    python tools/e2e_packed.py [--out DIR] [--nrec N]

(a) the pinned-record pipeline (the method of bench.py's e2e): cdfmoc_gpu_submit / _fetch over 3 slots, float32 records and
    int16 records alternating, both as raw big-endian file bytes (K3 swap, K3b unpack + swap); cells/s, H2D GB/s, share of
    cdfgpu_h2d_probe's ceiling; then, in a traced run of its own, the device time of the K3b and K3 kernels (torch.profiler).
(b) the cdfmoc_gpu command-line twin on a float and a packed gridV.nc on tmpfs: the record-loop phase ($CDFGPU_TIMING).
(c) the host decode the packed record needed before (nc3::Reader::read_f32), and read_raw of both records, on this host.
Prints one JSON line (and writes it to DIR/e2e_packed.json with --out).  Needs a GPU: there is no CPU fallback.
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

HBM_COPY_PEAK_GBS = 6545.6   # device-to-device copy peak the project measures its kernels against (DESIGN.md section 4)
SF, AO, SP = 1.0e-4, 0.0, -32768


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or ["?, ?"])[0].split(",", 1)
    return {"gpu": name.strip(), "power_limit": power.strip()}


def quantize(v, land):
    raw = np.clip(np.rint(v.astype(np.float64) / SF), -32767, 32767).astype(np.int16)
    raw[land] = SP
    return raw


def pipeline(lib, m, nrec):
    from cdftools_b200 import synth
    nk = m.nz - 1
    n3 = nk * m.ny * m.nx
    ib = synth.setup_masks(m)
    nz, ny, nb = lib.cdfmoc_setup(m.e1v, synth.setup_e3v_masked(m), ib)
    land = m.vmask[:-1] == 0
    hosts = {"f32": [], "i16": []}
    for r in range(3):
        raw = quantize(synth.make_v_record(m, r)[:-1], land)
        dec = raw.astype(np.float32) * np.float32(SF)
        dec[land] = SP
        for kind, a in (("f32", dec), ("i16", raw)):
            p = lib.PinnedArray(a.shape, a.dtype)
            p.array[...] = a.byteswap()   # raw big-endian file bytes
            hosts[kind].append(p)
    res = np.empty((3, nz, ny, nb))
    lib.set_input_big_endian(True)

    def use(kind):
        if kind == "i16":
            lib.set_input_packing(lib.FIELD_ZV, lib.INPUT_I16, SF, AO, SP)
        else:
            lib.set_input_packing(lib.FIELD_ZV, lib.INPUT_F32)

    def step(kind):
        pend = []
        for jt in range(nrec):
            s = jt % 3
            if len(pend) == 3:
                p0 = pend.pop(0)
                lib.cdfmoc_fetch(p0, res[p0])
            lib.cdfmoc_submit(s, jt, hosts[kind][jt % 3].array)
            pend.append(s)
        for s in pend:
            lib.cdfmoc_fetch(s, res[s])

    ceiling = lib.h2d_probe(hosts["f32"][0], reps=6)
    times = {"f32": [], "i16": []}
    for kind in ("f32", "i16"):   # warm-up of both paths (staging buffers, module load)
        use(kind)
        step(kind)
    for _ in range(3):            # alternating, same process
        for kind in ("f32", "i16"):
            use(kind)
            lib.synchronize()
            t0 = time.perf_counter()
            step(kind)
            lib.synchronize()
            times[kind].append(time.perf_counter() - t0)
    out = {"grid": "ORCA025 L75 (%d x %d x %d)" % (m.nx, m.ny, m.nz), "records_per_step": nrec, "h2d_ceiling_gbs": ceiling}
    for kind, es in (("f32", 4), ("i16", 2)):
        dt = min(times[kind])
        gbs = nrec * n3 * es / dt / 1e9
        out[kind] = {"ms_per_step": dt * 1e3, "ms_per_step_all": [t * 1e3 for t in times[kind]],
                     "cells_per_s": nrec * n3 * m.nz / nk / dt, "h2d_bytes_per_record": n3 * es,
                     "h2d_gbs": gbs, "frac_of_h2d_ceiling": gbs / ceiling}

    # device time of the input kernels, from a traced run of its own
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        kern = {}
        for kind, name in (("i16", "unpack_i16_kernel"), ("f32", "bswap32_kernel")):
            use(kind)
            lib.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                step(kind)
                lib.synchronize()
                torch.cuda.synchronize()
            d = [e.device_time for e in prof.events() if name in e.name and e.device_time > 0]   # microseconds
            if d:
                ms = float(np.median(d)) / 1e3
                nbytes = n3 * (6 if kind == "i16" else 8)
                kern[name] = {"ms_per_record": ms, "launches": len(d), "bytes_per_record": nbytes,
                              "gbs": nbytes / (ms * 1e-3) / 1e9, "frac_of_copy_peak": nbytes / (ms * 1e-3) / 1e9 / HBM_COPY_PEAK_GBS}
            else:
                kern[name] = "not measured (no such kernel in the trace)"
        out["input_kernels"] = kern
    except Exception as e:   # the timing above stands without the trace
        out["input_kernels"] = "not measured (%s)" % e
    use("f32")
    lib.set_input_big_endian(False)
    lib.cdfmoc_teardown()
    for ps in hosts.values():
        for p in ps:
            p.free()
    return out


_READ_TIMER = r"""
#include <chrono>
#include "nc3.hpp"
int main(int argc, char **argv)
{
    nc3::Reader r;
    if (!r.open(argv[1])) return 1;
    const nc3::Var &v = r.vars[r.find_var(argv[2])];
    const size_t n = (size_t)atol(argv[3]);
    std::vector<float> buf(n);
    double best_f32 = 1e30, best_raw = 1e30;
    for (int it = 0; it < 4; ++it) {
        auto t0 = std::chrono::steady_clock::now();
        if (!r.read_f32(v, 0, 0, n, buf.data())) return 1;
        auto t1 = std::chrono::steady_clock::now();
        if (!r.read_raw(v, 0, 0, n, buf.data())) return 1;
        auto t2 = std::chrono::steady_clock::now();
        if (it) {
            best_f32 = std::min(best_f32, std::chrono::duration<double>(t1 - t0).count());
            best_raw = std::min(best_raw, std::chrono::duration<double>(t2 - t1).count());
        }
    }
    printf("%.6f %.6f\n", best_f32, best_raw);
    return 0;
}
"""


def write_gridv(path, m, nrec, packed):
    from scipy.io import netcdf_file
    from cdftools_b200 import synth
    f = netcdf_file(str(path), "w", version=2)
    f.createDimension("time_counter", None)
    for n, l in (("x", m.nx), ("y", m.ny), ("depthv", m.nz)):
        f.createDimension(n, l)
    tc = f.createVariable("time_counter", "d", ("time_counter",))
    v = f.createVariable("vomecrty", "h" if packed else "f", ("time_counter", "depthv", "y", "x"))
    if packed:
        v.scale_factor = np.float32(SF)
        v.missing_value = np.int16(SP)
    else:
        v.missing_value = np.float32(SP)
    land = m.vmask == 0
    for r in range(nrec):
        tc[r] = 432000.0 * (r + 0.5)
        raw = quantize(synth.make_v_record(m, r % 3), land)
        if packed:
            v[r] = raw
        else:
            dec = raw.astype(np.float32) * np.float32(SF)
            dec[land] = SP
            v[r] = dec
    f.close()


def files(m, nrec):
    from cdftools_b200 import build, ncfiles
    out = {}
    n3 = (m.nz - 1) * m.ny * m.nx
    with tempfile.TemporaryDirectory() as bindir, \
            tempfile.TemporaryDirectory(dir="/dev/shm" if Path("/dev/shm").exists() else None) as d:
        tools = build.build_host(bindir=bindir, names=["cdfmoc_gpu"])
        timer = Path(bindir) / "read_timer"
        (Path(bindir) / "read_timer.cpp").write_text(_READ_TIMER)
        subprocess.run(["g++", "-O2", "-std=c++17", "-pthread", "-ffp-contract=off", "-I", str(ROOT / "cdftools_b200" / "csrc" / "host"),
                        "-o", str(timer), str(Path(bindir) / "read_timer.cpp")], check=True)
        d = Path(d)
        for kind in ("float", "packed"):
            (d / kind).mkdir()
            ncfiles.write_mesh(m, d / kind)
            write_gridv(d / kind / "gridV.nc", m, nrec, kind == "packed")
        # (c) host side of one record, page cache warm
        for kind in ("float", "packed"):
            t = subprocess.run([str(timer), str(d / kind / "gridV.nc"), "vomecrty", str(n3)], capture_output=True, text=True, check=True)
            f32, raw = map(float, t.stdout.split())
            out["host_read_%s" % kind] = {"read_f32_s": f32, "read_raw_s": raw}
        # (b) the command-line twin, alternating float / packed
        env = dict(os.environ, CDFGPU_TIMING="1")
        rec = {"float": [], "packed": []}
        for it in range(3):
            for kind in ("float", "packed"):
                r = subprocess.run([str(tools["cdfmoc_gpu"]), "-v", "gridV.nc"], cwd=d / kind, check=True, capture_output=True, text=True,
                                   env=env)
                ph = {l.split()[2]: float(l.split()[3]) for l in r.stderr.splitlines() if l.startswith("cdfmoc_gpu: phase")}
                if it:   # the first round warms the page cache
                    rec[kind].append(ph["records"])
            same = (d / "float" / "moc.nc").read_bytes() == (d / "packed" / "moc.nc").read_bytes()
        out["cli_records_phase_s"] = {k: min(v) for k, v in rec.items()}
        out["cli_records_phase_s_all"] = rec
        out["cli_records"] = nrec
        out["cli_gridv_bytes"] = {k: (d / k / "gridV.nc").stat().st_size for k in ("float", "packed")}
        out["cli_outputs_byte_identical"] = same
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--nrec", type=int, default=12)
    ap.add_argument("--file-records", type=int, default=8)
    a = ap.parse_args()
    from cdftools_b200 import lib, synth
    res = {"tool": "tools/e2e_packed.py", **card()}
    m = synth.make_mesh("ORCA025")
    lib.init(0, 3)
    try:
        res["pipeline"] = pipeline(lib, m, a.nrec)
    finally:
        lib.finalize()
    res["files"] = files(m, a.file_records)
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).mkdir(parents=True, exist_ok=True)
        (Path(a.out) / "e2e_packed.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
