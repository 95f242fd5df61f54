#!/usr/bin/env python3
"""bench.py -- MOC cells/s of the cdfmoc / cdfmocsig hot path on B200 (BASELINE.json metric), with roofline and
CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

--dump-outputs DIR writes what the timed kernel phase computed in its last step, DIR/cdfmoc.npy (record, level, j, basin) or
DIR/cdfmocsig.npy (record, j, bin, basin), fp64, so that two builds can be compared output for output: the inputs are
generated on the device from a fixed seed.  When the whole result exceeds 60 MB, a fixed seeded sample of whole records is
written; the JSON line lists which.  Single-process runs of --impl ours only.

Default workload (N=1, BASELINE.json configs[1]): cdfmoc on a synthetic ORCA025 L75 grid (1442x1021x75), 73 five-day
gridV records, 5 basins.  One STEP = one pass of the hot path over the whole record set of the workload.
  value : whole-job cells/s (rec*nx*ny*nz / t), records already resident in HBM (kernel phase)
  e2e   : the same job through the C-ABI record pipeline (cdf*_gpu_submit / cdf*_gpu_fetch) from pinned HOST
          buffers: H2D of every record and D2H of every result slab inside the timed region
  roofline : the workload's kernel (K1 moc_zonal_scan or K2 mocsig_eos_hist_scan): algorithmic bytes per launch /
          average launch time (CUDA events on the launch stream) against the measured HBM copy bandwidth
  cpu_baseline : the CPU restatement of the reference loops (oracle/, OpenMP over jj like the reference) on the
          box's host cores, bounded sample -- a reported baseline, not the target.  gfortran/netcdf are absent from
          this image, so the reference binary itself cannot be built (kind = "port").
N > 1: one process per GPU (torchrun).
  time sharding  (cdfmoc workloads, cdfmocsig-ORCA025): every rank owns its own records -> weak scaling
  band sharding  (cdfmocsig-ORCA12-...-bands): every rank owns a latitude band of every record -> strong scaling
Inside the timed region the per-rank result slabs are gathered to rank 0's HBM over NCCL behind their kernels (--gather
nccl, the default; cdftools_b200/shard.py); --gather host makes every rank copy its own slabs to page-locked host memory
instead (no collective at all -- faster at 2 GPUs, host-memory bound at 8); the other mode is measured in a sub-record.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree, which may be read-only

WORKLOADS = {
    "cdfmoc-ORCA025-L75-73rec-5basins": dict(kernel="moc", grid="ORCA025", nrec=73, shard="time"),
    "cdfmoc-ORCA2-L31-12rec-5basins": dict(kernel="moc", grid="ORCA2", nrec=12, shard="time"),
    "cdfmoc-ORCA12-L75-46rec-5basins": dict(kernel="moc", grid="ORCA12", nrec=46, shard="time"),
    "cdfmocsig-ORCA025-L75-sigma0-104bins-73rec": dict(kernel="sig", grid="ORCA025", nrec=73, shard="time",
                                                       pref=0.0, bins=(23.0, 0.05, 104)),
    "cdfmocsig-ORCA12-L75-sigma2-158bins-8rec-bands": dict(kernel="sig", grid="ORCA12", nrec=8, shard="band",
                                                           pref=2000.0, bins=(30.0, 0.05, 158)),
}
DEFAULT_WORKLOAD = "cdfmoc-ORCA025-L75-73rec-5basins"
METRIC = "MOC cells/s (rec*nx*ny*nz)"
ALL_CPUS = os.sched_getaffinity(0)   # before any binding


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed regions run."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.25)
            self.proc.terminate()
            self.thr.join(timeout=2)

    def summary(self):
        ok = [r for r in self.rows if len(r) >= 9]
        sm = [float(r[1]) for r in ok if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in ok if r[2].replace(".", "").isdigit()]
        pw = [float(r[3]) for r in ok if r[3].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[5 + i].lower().startswith("active") for r in ok)]
        # samples taken while the GPU was drawing power (the timed regions), if any
        hot = [s for s, p in zip(sm, pw) if p > 0.5 * max(pw)] if pw and len(pw) == len(sm) else sm
        return {"sm_mhz": float(np.median(hot or sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ------------------------------------------------------------------------------------------------ case construction
def build_case(spec, rows=None):
    from cdftools_b200 import synth   # (the oracle is not needed to build inputs: it is imported by the checker legs only)
    m = synth.make_mesh(spec["grid"], rows=rows)
    ib = synth.setup_masks(m)
    e3m = synth.setup_e3v_masked(m) if spec["kernel"] == "moc" else None
    return m, ib, e3m


def oracle_record(spec, m, ib, e3m, arrs, rows=None):
    """CPU oracle on one record (optionally a row subset).  For cdfmocsig the oracle skips the first and last row of
    what it is given, so callers hand it windows with a halo."""
    import oracle
    if spec["kernel"] == "moc":
        sl = slice(None) if rows is None else rows
        return oracle.cdfmoc_record(m.e1v[sl], e3m[:, sl], ib[sl], np.ascontiguousarray(arrs[0][:, sl]))
    smin, sstp, nbins = spec["bins"]
    sl = slice(None) if rows is None else rows
    out, _ = oracle.cdfmocsig_record(m.e1v[sl], m.e3v_0[:, sl], ib[sl], *(np.ascontiguousarray(a[:, sl]) for a in arrs),
                                     0.0, 0.0, 0.0, spec["pref"], 0, smin, sstp, nbins, want_bins=False)
    return out


def host_records(spec, m, n):
    from cdftools_b200 import synth
    recs = []
    for r in range(n):
        v = synth.make_v_record(m, r)[:-1]
        if spec["kernel"] == "moc":
            recs.append((v,))
        else:
            t, s = (x[:-1] for x in synth.make_ts_record(m, r))
            recs.append((v, t, s))
    return recs


DUMP_BYTES = 60_000_000


def dump_outputs(d: Path, name: str, out, n_res: int) -> dict:
    """--dump-outputs: the (nrec, ...) fp64 result of the last timed step as d/<name>.npy -- every record if they fit in
    DUMP_BYTES, else a sample of whole records drawn with a fixed seed (the same for the same workload)."""
    nrec = out.shape[0]
    k = max(1, min(nrec, DUMP_BYTES // (out[0].numel() * out.element_size())))
    pick = np.sort(np.random.default_rng(0).choice(nrec, k, replace=False))
    arr = out[pick.tolist()].cpu().numpy()
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / f"{name}.npy", arr)
    return {"dir": str(d), name: {"records": pick.tolist(), "of_records": nrec, "resident_records": n_res,
                                  "shape": list(arr.shape), "dtype": str(arr.dtype)}}


def use_all_host_cores():
    """The CPU arms use every host core: undo the GPU-local CPU binding and the OMP_NUM_THREADS=1 that torchrun exports."""
    import oracle
    try:
        os.sched_setaffinity(0, ALL_CPUS)
    except Exception:
        pass
    oracle.set_num_threads(len(ALL_CPUS))
    return oracle.num_threads()


def cpu_baseline(spec, m, ib, e3m, budget_s=15.0, max_rec=6):
    """Oracle port timed on the host cores (OpenMP over jj, as src/cdfmoc.f90:369 / cdfmocsig.f90:413)."""
    cores = use_all_host_cores()
    arrs = host_records(spec, m, 1)[0]
    t0 = time.perf_counter()
    oracle_record(spec, m, ib, e3m, arrs)
    t1 = time.perf_counter() - t0
    n = int(max(1, min(max_rec, budget_s / max(t1, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(n):
        oracle_record(spec, m, ib, e3m, arrs)
    dt = (time.perf_counter() - t0) / n
    cells = m.nx * m.ny * m.nz
    what = ("C restatement of src/cdfmoc.f90:352-388" if spec["kernel"] == "moc" else
            "C restatement of src/cdfmocsig.f90:366-475 + eos.f90:842-882, direct-scatter form (the reference's dense "
            "nb*nbins*nx pass per (j,k), cdfmocsig.f90:435-442, is several times slower)")
    return {"value": cells / dt, "unit": "cells/s", "cores": cores, "kind": "port",
            "sample": f"{n} record(s) of the same grid, compute only (arrays in RAM), {dt * 1e3:.1f} ms/record; "
                      f"{what}, gcc -O3 -ffp-contract=off -fopenmp, {cores} OpenMP threads"}


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    spec = WORKLOADS[args.workload]
    m, ib, e3m = build_case(spec)
    cores = use_all_host_cores()   # explicitly: under torchrun OMP_NUM_THREADS=1 would leave the port single-threaded
    cells = m.nx * m.ny * m.nz
    arrs = host_records(spec, m, 1)[0]
    t0 = time.perf_counter()
    oracle_record(spec, m, ib, e3m, arrs)
    t1 = time.perf_counter() - t0
    per_step = int(max(1, min(spec["nrec"], 4.0 / max(t1, 1e-3))))   # bounded sample: ~4 s of host time per step
    for _ in range(args.warmup):
        oracle_record(spec, m, ib, e3m, arrs)
    t0 = time.perf_counter()
    for _ in range(args.steps * per_step):
        oracle_record(spec, m, ib, e3m, arrs)
    dt = time.perf_counter() - t0
    val = cells * per_step * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "cells/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak" if spec["shard"] == "time" else "strong", "vs_baseline": None,
            "dtype": "f32 products, f64 sums", "data": "synthetic",
            "config": {"workload": args.workload, "grid": spec["grid"], "records_per_step": per_step,
                       "host_cpus": len(ALL_CPUS), "omp_threads": cores,
                       "note": "host CPU only; gfortran/netcdf absent so the reference binary cannot be built: this is "
                               "the C restatement of the reference loops with the reference's OpenMP directives"},
            "cpu_baseline": {"value": val, "unit": "cells/s", "cores": cores, "kind": "port",
                             "sample": f"{per_step} record(s) per step x {args.steps} steps, compute only, {cores} OpenMP threads"},
            "e2e": {"value": val, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def bind_to_gpu_numa_node(index: int):
    """Pin this rank's threads to the CPUs NVML reports as local to its GPU, BEFORE the pinned host buffers are allocated:
    with first-touch placement the record buffers then sit on the NUMA node of the GPU's PCIe root, so N ranks stream
    from N memory controllers instead of all from the node the launcher happened to start on.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        cpus = sorted(os.sched_getaffinity(0))
        pynvml.nvmlShutdown()
        return {"cpus": "%d-%d" % (cpus[0], cpus[-1]) if cpus else "", "n": len(cpus)}
    except Exception as e:   # no NVML / not permitted: run unbound
        return {"error": str(e)[:80]}


# ------------------------------------------------------------------------------------------------------- our arm
class Ctx:
    """What every measurement of this process shares."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from cdftools_b200 import lib, shard
        self.torch, self.dist, self.lib, self.shard, self.args = torch, dist, lib, shard, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device -- libcdfgpu has no CPU fallback")
        torch.cuda.set_device(self.local)
        self.numa = bind_to_gpu_numa_node(self.local)
        if self.world > 1:
            # the slab gather is small next to the kernels' traffic: a few NCCL channels keep it off the SMs the persistent
            # kernels occupy (each channel is a resident CTA)
            if args.spare_sms >= 0:
                os.environ["CDFGPU_K1_SPARE_SMS"] = str(args.spare_sms)
            if args.nccl_channels > 0:
                os.environ.setdefault("NCCL_MAX_NCHANNELS", str(args.nccl_channels))
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        lib.init(self.local, 3)
        lib.set_device_inputs_ready(True)   # records are resident and synchronised before the timed launches
        self.t_start = time.perf_counter()
        self.hbm_peak, self.peak_src = peaks()

    def elapsed(self):
        return time.perf_counter() - self.t_start

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())


def measure(cx: Ctx, workload: str, steps: int, warmup: int, nrec=None, do_e2e=True, do_smooth=True, do_cpu=False,
            clocks=None, gather=None, dump=None):
    """One workload on this process' GPU (all ranks call it together): kernel phase with the result slabs leaving the device
    (--gather), roofline,
    optional end-to-end pipeline, parity spot check against the oracle on rank 0.  Returns the JSON-able record (rank 0
    holds the meaningful one).  dump: directory for dump_outputs() of the kernel phase's last step."""
    torch, dist, lib, shard, args = cx.torch, cx.dist, cx.lib, cx.shard, cx.args
    rank, world = cx.rank, cx.world
    spec = WORKLOADS[workload]
    sig = spec["kernel"] == "sig"
    band = spec["shard"] == "band"
    from cdftools_b200 import synth
    nxg, nyg, nzg = synth.GRIDS[spec["grid"]]
    bands = shard.band_plan(nyg, world)
    j0, j1 = bands[rank] if band else (0, nyg)
    m, ib, e3m = build_case(spec, rows=(j0, j1) if band else None)
    nx, ny, nz, nb = m.nx, m.ny, m.nz, ib.shape[2]
    nrec = spec["nrec"] if nrec is None else min(nrec, spec["nrec"])
    cells_rec_local = nx * ny * nz
    cells_step_global = (nrec * nxg * nyg * nzg) if band else (world * nrec * cells_rec_local)
    if sig:
        smin, sstp, nbins = spec["bins"]
        lib.cdfmocsig_setup(m.e1v, m.e3v_0, ib, nz, nbins, smin, sstp, spec["pref"], lib.EOS80,
                            j_first_global=j0, ny_global=nyg)
        mxrows = max(b1 - b0 for b0, b1 in bands) if band else ny
        out_shape = (mxrows, nbins, nb)          # a band's slab is padded to the largest band: equal slabs for the gather
        bytes_launch = (nz - 1) * ny * nx * 16 + ny * nx * 1 + nb * nbins * ny * 8
        kname = "mocsig_eos_hist_scan_kernel"
    else:
        lib.cdfmoc_setup(m.e1v, e3m, ib)
        out_shape = (nz, ny, nb)
        bytes_launch = (nz - 1) * ny * nx * 8 + ny * nx * 1 + nb * ny * nz * 8
        kname = "moc_zonal_scan_kernel<%d>" % nb
    narr = 3 if sig else 1

    # ---- device-resident records (kernel phase).  Distinct records; together far larger than the 126 MB L2.
    gen = torch.Generator(device="cuda")
    gen.manual_seed(20261017 + rank)
    rec_bytes = (nz - 1) * ny * nx * 4 * narr
    free_b, total_b = torch.cuda.mem_get_info()
    # record r reads resident record r % n_res: for --dump-outputs n_res follows from the device, not from what other processes
    # hold at the moment, so that the same arguments give the same inputs
    n_res = int(max(2, min(nrec, ((total_b if dump is not None else free_b) * 0.55) // rec_bytes)))
    shape3 = (nz - 1, ny, nx)
    vmask = torch.from_numpy(m.vmask[:-1].astype(np.float32)).cuda()
    tmask = tbase = sbase = None
    if sig:
        tmask = torch.from_numpy(m.tmask[:-1].astype(np.float32)).cuda()
        z = torch.from_numpy(m.gdept_1d[:-1].astype(np.float32)).cuda()[:, None, None]
        cl = torch.cos(torch.deg2rad(torch.from_numpy(m.gphiv).cuda()))[None]
        tbase = (1.0 + 24.0 * torch.exp(-z / 1000.0) * cl ** 2)
        sbase = (34.2 + 1.2 * cl * torch.exp(-z / 600.0) + 0.5 * (1 - torch.exp(-z / 1500.0)))
    recs = []
    for r in range(n_res):
        v = torch.randn(shape3, device="cuda", generator=gen, dtype=torch.float32).mul_(0.1).mul_(vmask)
        if sig:   # same stratified, meridionally varying T/S as synth.make_ts_record, white noise 0.15 K
            t = (tbase + args.ts_noise * torch.randn(shape3, device="cuda", generator=gen) + 0.5 * np.sin(0.3 * r)).mul_(tmask)
            s = (sbase + 0.2 * args.ts_noise * torch.randn(shape3, device="cuda", generator=gen)).mul_(tmask)
            recs.append((v, t.float().contiguous(), s.float().contiguous()))
        else:
            recs.append((v,))
    del vmask
    outs = [torch.zeros((nrec,) + out_shape, dtype=torch.float64, device="cuda") for _ in range(2)]
    st = torch.cuda.Stream()
    comm = torch.cuda.Stream()

    # ---- the slab gather to rank 0 (the only communication of the path): records go in a few groups, each group's
    # slabs right behind its kernels on a side stream, into receive buffers allocated ONCE -- only the last group of the
    # last step is not overlapped by kernels
    ngroups = 1 if world == 1 else max(1, min(args.gather_groups, nrec // 2))
    gather = gather or args.gather
    do_gather = world > 1 and gather == "nccl"
    do_host = world > 1 and gather == "host"
    gb = [(g * nrec) // ngroups for g in range(ngroups + 1)]
    recv, full = None, None
    # What travels is what the writer needs: the output files hold REAL(4) (src/cdfmoc.f90:520-551 REAL(dmoc(...)) and the
    # derived inp0 = REAL(glo - atl); src/cdfmocsig.f90:478-483), so the slabs are converted on the device (fp64 difference
    # first, then the rounding, as the reference does) and half the bytes cross NVLink.  --gather-dtype f64 sends them raw.
    g32 = args.gather_dtype == "f32"
    nvar = (nb + 1 if (not sig and nb >= 5) else nb) if g32 else nb
    gshape = out_shape[:-1] + (nvar,)
    gdtype = torch.float32 if g32 else torch.float64
    gmax = max(gb[g + 1] - gb[g] for g in range(ngroups))
    send = torch.empty((gmax,) + gshape, dtype=gdtype, device="cuda") if (do_gather and g32) else None
    if do_gather and rank == 0:
        recv = [torch.empty((gmax,) + gshape, dtype=gdtype, device="cuda") for _ in range(world)]
        if band:
            full = torch.empty((nrec, nyg) + gshape[1:], dtype=gdtype, device="cuda")
    # --gather host (default): no collective at all.  The result is a file, so rank 0 need not hold the slabs in HBM: every
    # rank copies its own slabs to page-locked host memory (copy engine, no SMs) right behind their kernels.
    hres = [torch.empty((nrec,) + out_shape, dtype=torch.float64, pin_memory=True) for _ in range(2)] if do_host else None

    def launch(rec, o):
        if sig:
            lib.cdfmocsig_compute_device(rec[0], rec[1], rec[2], o, stream=st)
        else:
            lib.cdfmoc_compute_device(rec[0], o, st)

    diff64 = torch.empty((gmax,) + out_shape[:-1], dtype=torch.float64, device="cuda") if (do_gather and g32 and nvar > nb) else None
    gathered = [None, None]   # per output buffer: the event that marks its last gather as complete

    # cdfmoc: the records of a group go to the device as ONE persistent launch (cdfmoc_gpu_compute_device_batch: the work
    # units run over (record, row, levels), so launch overhead, ramp-up and tail are paid once per group) unless
    # --k1-launch record asks for one launch per record (what the submit / fetch record pipeline issues)
    k1_batch = (not sig) and args.k1_launch == "batch"
    zlists = [[recs[r % n_res][0] for r in range(gb[g], gb[g + 1])] for g in range(ngroups)]
    olists = [[[outs[b][r] for r in range(gb[g], gb[g + 1])] for g in range(ngroups)] for b in range(2)]

    def kernel_step(i):
        o = outs[i & 1]
        if gathered[i & 1] is not None:
            st.wait_event(gathered[i & 1])   # this buffer's slabs of two steps ago must have left before it is overwritten
        for g in range(ngroups):
            with torch.cuda.stream(st):
                if k1_batch:
                    lib.cdfmoc_compute_device_batch(zlists[g], olists[i & 1][g], st)
                else:
                    for r in range(gb[g], gb[g + 1]):
                        launch(recs[r % n_res], o[r])
            if do_host:
                ev = torch.cuda.Event()
                ev.record(st)
                with torch.cuda.stream(comm):
                    comm.wait_event(ev)
                    hres[i & 1][gb[g]:gb[g + 1]].copy_(o[gb[g]:gb[g + 1]], non_blocking=True)
            if do_gather:
                ev = torch.cuda.Event()
                ev.record(st)
                with torch.cuda.stream(comm):
                    comm.wait_event(ev)
                    part = o[gb[g]:gb[g + 1]]
                    if g32:   # output conversion on the device: REAL(psi), and inp0 = REAL(psi_glo - psi_atl) for cdfmoc
                        p32 = send[: part.shape[0]]
                        p32[..., :nb].copy_(part)
                        if nvar > nb:
                            torch.sub(part[..., 0], part[..., 1], out=diff64[: part.shape[0]])
                            p32[..., nb].copy_(diff64[: part.shape[0]])
                        part = p32
                    dist.gather(part, [b[: part.shape[0]] for b in recv] if rank == 0 else None, dst=0)
                    if band and rank == 0:   # unpack the padded bands into the (record, j, bin, basin) array the writer wants
                        for rr, (b0, b1) in enumerate(bands):
                            full[gb[g]:gb[g + 1], b0:b1].copy_(recv[rr][: part.shape[0], : b1 - b0])
        if do_gather or do_host:
            gathered[i & 1] = torch.cuda.Event()
            gathered[i & 1].record(comm)

    def sync_all():
        st.synchronize()
        comm.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for i in range(warmup):
        kernel_step(i)
    sync_all()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = lib.launch_count()
    ev0.record(st)
    for i in range(steps):
        kernel_step(i)
    if world > 1:
        st.wait_stream(comm)   # the timed region ends when the last gather has landed on rank 0
    ev1.record(st)
    sync_all()
    launches = lib.launch_count() - l0
    # before anything below reuses the output buffers or the resident records
    dumped = dump_outputs(dump, "cdfmocsig" if sig else "cdfmoc", outs[(steps - 1) & 1], n_res) if dump is not None and rank == 0 else None
    ms_total = cx.max_over_ranks(ev0.elapsed_time(ev1))
    ms_step = ms_total / steps
    value = cells_step_global / (ms_step * 1e-3)

    # ---- roofline of the workload's kernel: algorithmic bytes per launch / average launch time (same events)
    hbm_peak = cx.hbm_peak
    ms_record = ms_total / (steps * nrec)
    achieved = bytes_launch / (ms_record * 1e-3) / 1e9
    rpl = nrec / ngroups if k1_batch else 1.0          # records per launch
    ms_launch = ms_record * rpl
    roofline = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "traffic": None, "kernel": kname, "bytes_per_launch": int(bytes_launch * rpl), "ms_per_launch": ms_launch,
                "records_per_launch": rpl, "bytes_per_record": bytes_launch, "ms_per_record": ms_record,
                "peak_source": cx.peak_src, "frac_of_8TBps_spec": achieved / 8000.0,
                "note": "per-GPU figure; at N>1 the launch time includes the overlapped copy of the result slabs (--gather)",
                "peak_kind": "measured device-to-device COPY bandwidth (read + write); a read-only streaming kernel can "
                             "exceed it slightly (frac > 1) -- see frac_of_8TBps_spec"}
    tp = ROOT / "profiles" / ("k2_traffic.json" if sig else "k1_traffic.json")
    if tp.exists() and spec["grid"] == "ORCA025" and not band:
        try:
            tj = json.loads(tp.read_text())
            roofline["traffic"] = tj["dram_bytes_per_launch"] * rpl   # (the capture is one record)
            roofline["traffic_source"] = "committed ncu capture of this kernel on this grid (%s), not a counter of this run" % tp.name
            if sig and "warp_inst_per_launch" in tj:
                roofline["warp_inst_per_launch"] = tj["warp_inst_per_launch"]
        except Exception:
            pass

    # ---- end to end through the record pipeline: pinned host -> H2D (copy stream) -> kernel -> D2H
    e2e = None
    host, res = [], None
    if do_e2e:
        n_host = min(nrec, 6 if not sig else 3)
        host = [[lib.PinnedArray(shape3, np.float32) for _ in range(narr)] for _ in range(n_host)]
        for h, r in zip(host, (recs * n_host)[:n_host]):
            for ha, ra in zip(h, r):
                ha.array[...] = ra.cpu().numpy()
        eshape = (ny,) + out_shape[1:] if sig else out_shape
        res = lib.PinnedArray((3,) + eshape, np.float64)
        nslots = 3
        # the platform's ceiling for the input leg: all ranks copy pinned records to their GPUs at once, nothing else running
        if world > 1:
            dist.barrier()
        h2d_gbs = lib.h2d_probe(host[0][0], reps=6)
        h2d_all = cx.sum_over_ranks(h2d_gbs)

        def e2e_step():
            pend = []
            for jt in range(nrec):
                s = jt % nslots
                if len(pend) == nslots:
                    p0 = pend.pop(0)
                    (lib.cdfmocsig_fetch if sig else lib.cdfmoc_fetch)(p0, res.array[p0])
                h = host[jt % n_host]
                if sig:
                    lib.cdfmocsig_submit(s, jt, h[0].array, h[1].array, h[2].array)
                else:
                    lib.cdfmoc_submit(s, jt, h[0].array)
                pend.append(s)
            for s in pend:
                (lib.cdfmocsig_fetch if sig else lib.cdfmoc_fetch)(s, res.array[s])

        e2e_steps = max(1, min(steps, 3))
        e2e_step()
        lib.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        lib.synchronize()
        torch.cuda.synchronize()
        dt = cx.max_over_ranks(time.perf_counter() - t0)
        h2d_bytes = nrec * rec_bytes
        gbs_all = world * h2d_bytes * e2e_steps / dt / 1e9
        e2e = {"value": cells_step_global * e2e_steps / dt, "unit": "cells/s", "h2d_bytes_per_step": h2d_bytes,
               "d2h_bytes_per_step": nrec * int(np.prod(eshape)) * 8, "steps": e2e_steps,
               "ms_per_step": dt / e2e_steps * 1e3,
               "path": "cdf%s_gpu_submit/_fetch, 3 slots, pinned host records (per rank)" % ("mocsig" if sig else "moc"),
               "h2d_gbs_all_ranks": gbs_all,
               "h2d_ceiling_gbs_all_ranks": h2d_all,
               "frac_of_h2d_ceiling": gbs_all / h2d_all if h2d_all > 0 else None,
               "h2d_ceiling_note": "all ranks copying one pinned record to their GPU at once (cudaMemcpyAsync, no kernels): what "
                                   "this host's PCIe / memory system delivers; the pipeline is bound by it, not by the kernels",
               "cpu_affinity_rank0": cx.numa}

    # ---- parity spot check of the timed kernel against the oracle (sampled latitude rows of one record)
    parity = None
    if rank == 0:
        got_all = outs[(steps - 1) & 1][0].cpu().numpy()
        arrs = [a.cpu().numpy() for a in recs[0]]
        errs, ok = [], True
        cand = np.unique(np.linspace(1, ny - 2, 5).astype(int)) if ny > 4 else np.arange(ny)
        for jr in cand:
            if sig:
                w = slice(jr - 1, jr + 2)
                ref = oracle_record(spec, m, ib, e3m, arrs, rows=w)[1]
                got = got_all[jr]
            else:
                ref = oracle_record(spec, m, ib, e3m, arrs, rows=slice(jr, jr + 1))[:, 0]
                got = got_all[:, jr]
            d = np.abs(got - ref)
            errs.append(float(d.max()))
            ok = ok and bool(np.all(d <= np.maximum(1e-9 * np.abs(ref), 1e-6)))
        parity = {"rows_checked": int(len(cand)), "max_abs_err_sv": max(errs), "within_tolerance": ok,
                  "tolerance": "1e-9 relative or 1e-6 Sv"}
        if do_host:   # what landed in host memory is what the device holds
            torch.cuda.synchronize()
            parity["host_copy_equals_device"] = bool(torch.equal(hres[(steps - 1) & 1], outs[(steps - 1) & 1].cpu()))
        if band and full is not None:   # the gathered array on rank 0 holds every band: rank 0's own rows must be in place
            parity["gathered_equals_local"] = bool(torch.equal(full[0, j0:j1, :, :nb], outs[(steps - 1) & 1][0, : j1 - j0].to(gdtype)))

    # ---- cdfmocsig only: the same kernel on T/S as smooth as the stratification (no cell-to-cell noise), one untimed
    # and one timed pass over the resident records.  The headline `value` stays the white-noise case (worst case for the
    # density-class run merge); this shows the other end of the range.  Done last: it overwrites the resident T/S.
    if sig and do_smooth:
        for r, rec in enumerate(recs):
            rec[1].copy_((tbase + 0.5 * np.sin(0.3 * r)).mul_(tmask))
            rec[2].copy_(sbase * tmask)
        for i in range(2):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(st):
                e0.record(st)
                for r in range(nrec):
                    launch(recs[r % n_res], outs[0][r])
                e1.record(st)
            st.synchronize()
        ms_s = cx.max_over_ranks(e0.elapsed_time(e1)) / nrec
        ach_s = bytes_launch / (ms_s * 1e-3) / 1e9
        roofline["smooth_ts"] = {"ms_per_launch": ms_s, "achieved": ach_s, "frac": ach_s / hbm_peak,
                                 "note": "same launches with ts_noise = 0 (T/S as smooth as the stratification)"}
    filt = lib.cdfmocsig_filter_info() if sig else None

    # ---- cdfmoc only: the same records with the OTHER launch mode (no slab gather): one launch per record when the
    # headline is batched, one batched launch per step otherwise
    if not sig:
        o = outs[0]
        zl = [recs[r % n_res][0] for r in range(nrec)]
        ol = [o[r] for r in range(nrec)]
        for i in range(2):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(st):
                e0.record(st)
                for _ in range(3):
                    if k1_batch:
                        for r in range(nrec):
                            lib.cdfmoc_compute_device(zl[r], ol[r], st)
                    else:
                        lib.cdfmoc_compute_device_batch(zl, ol, st)
                e1.record(st)
            st.synchronize()
        ms_b = cx.max_over_ranks(e0.elapsed_time(e1)) / (3 * nrec)
        ach_b = bytes_launch / (ms_b * 1e-3) / 1e9
        same = bool(torch.equal(o[0], outs[1][0])) if steps > 1 else None
        roofline["per_record_launches" if k1_batch else "batched"] = {
            "ms_per_record": ms_b, "achieved": ach_b, "frac": ach_b / hbm_peak, "records_per_launch": 1 if k1_batch else nrec,
            "equals_headline_result": same,
            "note": ("cdfmoc_gpu_compute_device: one launch per record (programmatic dependent launch), what cdfmoc_gpu_submit issues"
                     if k1_batch else "cdfmoc_gpu_compute_device_batch: one persistent launch per step over all records")}

    cb = None
    if do_cpu and rank == 0 and world == 1:
        cb = cpu_baseline(spec, m, ib, e3m)
    rec = {"workload": workload, "value": value, "unit": "cells/s", "ms_per_step": ms_step, "steps": steps, "warmup": warmup,
           "scaling": "strong" if band else "weak", "roofline": roofline, "gpu_launches": int(launches),
           "parity_check": parity,
           "config": {"workload": workload, "grid": spec["grid"], "nx": nxg, "ny": nyg, "nz": nzg,
                      "basins": nb, "records_per_step_per_gpu": nrec, "resident_records": n_res, "rows_per_gpu": ny,
                      "l2": "inputs (%.1f GB resident per GPU) are far larger than the 126 MB L2; no flush needed"
                            % (n_res * rec_bytes / 1e9),
                      "sharding": (("latitude bands" if band else "time (each rank owns its own records)") +
                                   {"host": "; no collective", "nccl": " + NCCL slab gather", "none": ""}[gather])
                                  if world > 1 else "single GPU",
                      "gather": ("%d group(s) per step behind their kernels, %s slabs, preallocated receive buffers, "
                                 "NCCL_MAX_NCHANNELS=%s" % (ngroups, "REAL(4) output-ready" if g32 else "fp64",
                                                            os.environ.get("NCCL_MAX_NCHANNELS"))) if do_gather else
                                ("every rank copies its own fp64 slabs to page-locked host memory in %d group(s) per step behind "
                                 "their kernels, inside the timed region (the result is a file: no rank needs the others' slabs "
                                 "in HBM)" % ngroups) if do_host else
                                ("SKIPPED (--gather none diagnostic)" if world > 1 else None),
                      "launches": ("one persistent launch per %s (%d records): cdfmoc_gpu_compute_device_batch"
                                   % ("step" if ngroups == 1 else "gather group", int(round(rpl)))) if k1_batch else
                                  "one launch per record, programmatic dependent launch between them",
                      "wet_fraction": m.wet_fraction}}
    if e2e:
        rec["e2e"] = e2e
    if dumped:
        rec["dump_outputs"] = dumped
    if cb:
        rec["cpu_baseline"] = cb
    if sig:
        rec["config"].update({"pref": spec["pref"], "sigmin": spec["bins"][0], "sigstp": spec["bins"][1],
                              "nbins": spec["bins"][2], "eos": "EOS80 polynomial", "ts_noise_K": args.ts_noise,
                              "ts_noise": "white, cell to cell (0.15 K: every neighbour in another density class, the "
                                          "worst case for run merging; 0: as smooth as the stratification)",
                              "bin_function": filt})
    for h in host:
        for ha in h:
            ha.free()
    if res is not None:
        res.free()
    (lib.cdfmocsig_teardown if sig else lib.cdfmoc_teardown)()
    del recs, outs, recv, full, tmask, tbase, sbase
    torch.cuda.empty_cache()
    return rec


def issue_bound(cx: Ctx, k2: dict):
    """K2's second bound (BASELINE.md section 2: the arithmetic ceiling must be measured before K2 is called HBM-bound).
    The bin function runs in packed fp32, so the ceiling is instruction ISSUE: the kernel's warp-instructions per launch
    (committed ncu count) against the issue rate this device sustains on an fp32-FMA / integer mix, measured here."""
    mb = cx.lib.microbench()
    rl = k2["roofline"]
    out = {"microbench": mb,
           "note": "warp-instructions per clock and SM with 8 warps per scheduler and 8 independent chains per thread; "
                   "dfma = the fp64 pipe the reference-exact tiers use, ffma2 = the packed fp32 FMA of the fp32 tier"}
    wi = rl.get("warp_inst_per_launch")
    if wi:
        rate = mb["ffma_int_mix"]["ginst_per_s"] * 1e9
        ms_issue = wi / rate * 1e3
        ms_hbm = rl["bytes_per_launch"] / (cx.hbm_peak * 1e9) * 1e3
        out.update({"warp_inst_per_launch": wi, "issue_ms_per_launch": ms_issue, "hbm_ms_per_launch": ms_hbm,
                    "binding": "issue" if ms_issue > ms_hbm else "hbm",
                    "frac_of_min_bound": max(ms_issue, ms_hbm) / rl["ms_per_launch"],
                    "frac_of_min_bound_smooth": max(ms_issue, ms_hbm) / rl["smooth_ts"]["ms_per_launch"] if "smooth_ts" in rl else None})
    return out


def e2e_files(cx: Ctx, nrec=12):
    """End to end INCLUDING NetCDF I/O: a synthetic ORCA025 gridV file + mesh / mask files on tmpfs -> the cdfmoc_gpu
    command-line twin (a process of its own: CUDA start-up, mesh and mask read, setup, record pipeline, moc.nc)."""
    import tempfile
    from cdftools_b200 import build, ncfiles, synth
    m = synth.make_mesh("ORCA025")
    with tempfile.TemporaryDirectory() as bindir, \
            tempfile.TemporaryDirectory(dir="/dev/shm" if Path("/dev/shm").exists() else None) as d:
        tools = build.build_host(bindir=bindir, names=["cdfmoc_gpu"])   # outside the tree, which may be read-only
        ncfiles.write_mesh(m, d)
        ncfiles.write_gridv(m, Path(d) / "gridV.nc", nrec)
        size = (Path(d) / "gridV.nc").stat().st_size
        env = dict(os.environ, CDFGPU_DEVICE=str(cx.local))
        subprocess.run([tools["cdfmoc_gpu"], "-v", "gridV.nc"], cwd=d, check=True, capture_output=True, env=env)   # warm page cache
        env["CDFGPU_TIMING"] = "1"   # phase times on stderr
        t0 = time.perf_counter()
        r = subprocess.run([tools["cdfmoc_gpu"], "-v", "gridV.nc"], cwd=d, check=True, capture_output=True, env=env, text=True)
        dt = time.perf_counter() - t0
        phases = [l for l in (r.stderr or "").splitlines() if l.startswith("cdfmoc_gpu: phase")]
    cells = nrec * m.nx * m.ny * m.nz
    ph = {}
    for l in phases:   # "cdfmoc_gpu: phase <name> <seconds>"
        w = l.split()
        ph[w[2]] = float(w[3])
    steady = {"records_phase_s": ph["records"], "records_phase_cells_per_s": cells / ph["records"],
              "records_phase_file_gbs": size / ph["records"] / 1e9,
              "note": "the record loop alone (read -> pinned -> H2D -> swap -> K1 -> D2H -> write): what a long run converges to; "
                      "the rest of the wall clock is CUDA context creation (overlapped with the mesh / mask read) and the "
                      "driver's teardown of the process"} if ph.get("records") else None
    return {"tool": "cdfmoc_gpu -v gridV.nc", "grid": "ORCA025", "records": nrec, "gridV_bytes": size, "wall_s": dt,
            "value": cells / dt, "unit": "cells/s", "phases": ph, "steady_state": steady,
            "note": "whole process wall clock: CUDA init, mesh / mask files, setup, then fread of raw big-endian records -> "
                    "pinned -> H2D -> GPU byte swap -> K1 -> D2H -> moc.nc; files on tmpfs"}


def siblings(cx: Ctx):
    """The sibling kernels of SURVEY.md section 8 (f3) on one ORCA025 record each, through the C ABI with host arrays: device
    time of the kernels (events inside the library), algorithmic bytes / that time against the HBM peak.  K7 (cdfsigtrp) is a
    section, not a field: device time, wall time through the ABI, and equality with the oracle's result."""
    from cdftools_b200 import synth
    lib, peak = cx.lib, cx.hbm_peak
    m = synth.make_mesh("ORCA025")
    nk, ny, nx = m.nz - 1, m.ny, m.nx
    n3 = nk * ny * nx
    rng = np.random.default_rng(11)
    out = {}

    def rec(name, ms, nbytes, note):
        out[name] = {"ms_per_record": ms, "bytes_per_record": int(nbytes), "achieved_gbs": nbytes / (ms * 1e-3) / 1e9,
                     "frac": nbytes / (ms * 1e-3) / 1e9 / peak, "note": note}

    zv = synth.make_v_record(m, 3)[:nk].astype(np.float32)
    msk = m.tmask[:nk].astype(np.float32)
    zm = np.stack([msk[0], m.tmaskatl, np.minimum(1.0, m.tmaskind + m.tmaskpac), m.tmaskind, m.tmaskpac], -1).astype(np.float32)
    e2 = (m.e1v * np.float32(0.75)).astype(np.float32)
    shape = lib.cdfzonal_setup(m.e1v, e2, zm, msk)
    for _ in range(2):
        lib.cdfzonal_sum(zv, shape)
    rec("K4_cdfzonalsum", lib.cdfzonal_kernel_ms(), n3 * 8, "zv + level mask, 5 basins (src/cdfzonalsum.f90:309-322)")
    for _ in range(2):
        lib.cdfzonal_mean(zv, shape)
    rec("K4_cdfzonalmean", lib.cdfzonal_kernel_ms(), n3 * 8, "src/cdfzonalmean.f90:312-344")
    lib.cdfzonal_teardown()
    dims = lib.cdfmhst_setup(m.e1v, m.e3v_0, m.vmask[0].astype(np.float32), m.tmaskatl, m.tmaskpac, m.tmaskind)
    zvt = (synth.make_v_record(m, 4) * 10.0).astype(np.float32)
    zvs = (synth.make_v_record(m, 5) * 35.0).astype(np.float32)
    for _ in range(2):
        lib.cdfmhst_record(zvt, zvs, dims)
    rec("K5_cdfmhst", lib.cdfmhst_kernel_ms(), m.nz * ny * nx * 12, "vomevt + vomevs + e3v (src/cdfmhst.f90:303-366)")
    lib.cdfmhst_teardown()
    pref, nb, smin, scal, zoom, smn = lib.TRANSIG_CODES["1000"]
    _, _, itab, scm = lib.transig_bins(nb, smin, scal, zoom, smn)
    e2u = (m.e1u * np.float32(0.9)).astype(np.float32)
    e3u = (m.e3v_0 * np.float32(1.01)).astype(np.float32)
    lib.cdftransig_setup(e2u, m.e1v, e3u[:nk], m.e3v_0[:nk], m.nz, nb, pref, smin, scm, itab)
    zu = (synth.make_v_record(m, 6)[:nk] * m.umask[:nk]).astype(np.float32)
    zt, zs = (x[:nk] for x in synth.make_ts_record(m, 0))
    for i in range(2):
        lib.cdftransig_record(zu, zv * m.vmask[:nk], zt, zs, i == 0)
    rec("K6_cdftransig_xy3d", lib.cdftransig_kernel_ms(), n3 * 80, "src/cdftransig_xy3d.f90:396-461, 93 classes; about 80 bytes per "
        "level-cell (densities written and re-read, velocities, metrics, masks, two scattered fp64 read-modify-writes)")
    lib.cdftransig_teardown()
    # K7: a long section (an ORCA12 line across the Atlantic) in 100 classes
    import oracle
    sec = synth.make_section(4000, 75, seed=5)
    p = oracle.sigtrp_prepare(sec["gdept"][0], sec["e3w_a"], sec["e3w_b"], sec["zu"], 0.0, sec["zs_a"], sec["zs_b"], 0.0, sec["zt_a"],
                              sec["zt_b"])
    a = (sec["eu"], sec["de3"], p["ddepu"], sec["gdepw"], p["zu"], p["zt"], p["zs"], p["zmask"], p["nk"], 23.0, 28.5, 100)
    lib.cdfsigtrp_section(*a)
    t0 = time.perf_counter()
    got = lib.cdfsigtrp_section(*a)
    t_abi = time.perf_counter() - t0
    t0 = time.perf_counter()
    ref = oracle.sigtrp_section(*a)
    t_cpu = time.perf_counter() - t0
    out["K7_cdfsigtrp"] = {"section": "4000 columns x 75 levels, 100 classes", "kernels_ms": lib.cdfsigtrp_kernel_ms(),
                           "abi_call_ms": t_abi * 1e3, "oracle_ms": t_cpu * 1e3, "oracle_threads": oracle.num_threads(),
                           "equals_oracle": bool(all(np.array_equal(got[k], ref[k], equal_nan=True) for k in ref)),
                           "note": "src/cdfsigtrp.f90:559-627; O(columns x classes x levels) latency-bound work, not a roofline item "
                                   "(the ABI call copies every intermediate array back: dhiso, dwtrp, dwtrpbin)"}
    out["parity"] = "tests/test_gpu_siblings.py, tests/test_transig.py, tests/test_sigtrp.py (bit-exact classes; sums within 1e-12 relative)"
    return out


def run_ours(args):
    cx = Ctx(args)
    rank, world = cx.rank, cx.world
    with ClockSampler(cx.local) as clk:
        main = measure(cx, args.workload, args.steps, args.warmup, do_e2e=True, do_cpu=True, dump=args.dump_outputs)
    line = None
    if rank == 0:
        spec = WORKLOADS[args.workload]
        line = {"metric": METRIC, "value": main["value"], "unit": "cells/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True,
                "scaling": main["scaling"], "vs_baseline": None, "dtype": "f32 products, f64 sums", "data": "synthetic",
                "config": main["config"], "roofline": main["roofline"], "e2e": main.get("e2e"),
                "gpu_launches": main["gpu_launches"], "clocks": clk.summary(), "parity_check": main["parity_check"]}
        if "cpu_baseline" in main:
            line["cpu_baseline"] = main["cpu_baseline"]
        if "dump_outputs" in main:
            line["dump_outputs"] = main["dump_outputs"]

    # ---- sub-records: the other BASELINE.json configurations, each to the same parity + roofline bar, while the budget lasts
    subs = {}

    def sub(name, fn, need_s):
        if args.no_subrecords or args.workload != DEFAULT_WORKLOAD:
            return
        go = cx.elapsed() + need_s < args.budget_s
        if world > 1:   # every rank takes the same decision
            t = cx.torch.tensor([1.0 if go else 0.0], device="cuda", dtype=cx.torch.float64)
            cx.dist.all_reduce(t, op=cx.dist.ReduceOp.MIN)
            go = bool(t.item() > 0.5)
        if not go:
            subs[name] = {"skipped": "time budget (%.0f s used of %.0f)" % (cx.elapsed(), args.budget_s)}
            return
        try:
            subs[name] = fn()
        except Exception as e:   # a sub-record must never take the headline line down with it
            if world > 1:
                raise
            subs[name] = {"error": repr(e)[:300]}

    if world == 1:
        def k2():
            r = measure(cx, "cdfmocsig-ORCA025-L75-sigma0-104bins-73rec", steps=3, warmup=3, nrec=12, do_e2e=False)
            r["second_bound"] = issue_bound(cx, r)
            return r
        sub("k2_config3", k2, 60)
        sub("e2e_files", lambda: e2e_files(cx), 90)
        sub("siblings", lambda: siblings(cx), 60)
    else:
        sub("config4", lambda: measure(cx, "cdfmoc-ORCA12-L75-46rec-5basins", steps=3, warmup=3, nrec=6, do_e2e=False), 240)
        sub("config5", lambda: measure(cx, "cdfmocsig-ORCA12-L75-sigma2-158bins-8rec-bands", steps=3, warmup=3, nrec=4,
                                       do_e2e=False), 120)
        # the headline workload once more with the result slabs leaving the devices the other way
        other = "host" if args.gather == "nccl" else "nccl"
        sub("gather_" + other, lambda: measure(cx, args.workload, steps=min(args.steps, 5), warmup=3, do_e2e=False, do_smooth=False,
                                               gather=other), 60)
    if rank == 0:
        line["sub_records"] = subs
        line["wall_s"] = cx.elapsed()
        print(json.dumps(line))
    cx.lib.finalize()
    if world > 1:
        cx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=list(WORKLOADS))
    ap.add_argument("--ts-noise", type=float, default=0.15,
                    help="cdfmocsig workloads: amplitude (K) of the cell-to-cell white noise on T (x0.2 on S); 0.15 is the "
                         "worst case for density-class run merging, 0 gives fields as smooth as the stratification")
    ap.add_argument("--budget-s", type=float, default=420.0,
                    help="wall-clock budget of this process: a sub-record (the other BASELINE configurations) is only started "
                         "while its estimated duration still fits")
    ap.add_argument("--no-subrecords", action="store_true", help="headline workload only")
    ap.add_argument("--nccl-channels", type=int, default=0,
                    help="NCCL_MAX_NCHANNELS for the slab gather (unless already set); 0 leaves NCCL's default")
    ap.add_argument("--k1-launch", default="batch", choices=["batch", "record"],
                    help="cdfmoc workloads: batch = the records of a step (of a gather group at N>1) in one persistent launch "
                         "(cdfmoc_gpu_compute_device_batch); record = one launch per record")
    ap.add_argument("--spare-sms", type=int, default=-1,
                    help="N>1 with --gather nccl: SMs the persistent K1 grid leaves to the NCCL kernels ($CDFGPU_K1_SPARE_SMS); "
                         "-1 = the default for the mode")
    ap.add_argument("--gather-dtype", default="f32", choices=["f32", "f64"],
                    help="slabs gathered to rank 0: f32 = converted on the device to what the output file stores (REAL(4), plus "
                         "the derived inp0 for cdfmoc); f64 = the raw fp64 slabs")
    ap.add_argument("--gather-groups", type=int, default=4, help="the slabs of a step are gathered in this many groups")
    ap.add_argument("--gather", default="nccl", choices=["host", "nccl", "none"],
                    help="N>1, where the result slabs go inside the timed region: nccl = gathered to rank 0's HBM over NVLink "
                         "(default); host = every rank copies its own fp64 slabs to page-locked host memory (no collective; at "
                         "8 GPUs the 160 GB/s of result traffic saturate the host memory system); none = diagnostic, slabs stay "
                         "on the device (the number is then NOT the job's)")
    ap.add_argument("--dump-outputs", type=Path, default=None, metavar="DIR",
                    help="write the fp64 result of the last timed step (a fixed sample of its records above 60 MB) to "
                         "DIR/cdfmoc.npy or DIR/cdfmocsig.npy, after the workload's kernel; single-process runs of "
                         "--impl ours only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs: single-process runs of --impl ours only")
    if args.impl == "reference":
        run_reference(args)
    else:
        args.warmup = max(args.warmup, 3)
        run_ours(args)


if __name__ == "__main__":
    main()
