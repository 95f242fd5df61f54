/*
 * cdfgpu.h -- C ABI of libcdfgpu.so: the B200 (sm_100a) implementation of the CDFTOOLS meridional-overturning
 * hot path (cdfmoc zonal transport integral + vertical scan; cdfmocsig fused EOS + density-class scatter-add).
 *
 * The reference (meom-group/CDFTOOLS) is Fortran 90 with no FFI: each tool is a monolithic PROGRAM.  This ABI is
 * cut exactly around the two loop nests that are the hot path, so that a thin ISO_C_BINDING layer
 * (cdftools_b200/fortran/cdfgpu_mod.f90, INTEGRATION.md) can replace them in place:
 *
 *     src/cdfmoc.f90:352-388      -> cdfmoc_gpu_submit / cdfmoc_gpu_fetch
 *     src/cdfmocsig.f90:366-475   -> cdfmocsig_gpu_submit / cdfmocsig_gpu_fetch
 *
 * Conventions
 *   - Plain pointers and sizes only.  Every entry point returns 0 (CDFGPU_OK) or a CDFGPU_ERR_* code;
 *     cdfgpu_last_error() holds the text.  The Fortran host does `IF (ierr /= 0) STOP 97`.
 *   - Arrays are passed in the reference's own memory order (Fortran column-major == C [k][j][i]):
 *       e1v(nx,ny) REAL(4), e3v(nx,ny,nz) REAL(4), ibmask(nb,nx,ny) INTEGER(2) basin fastest,
 *       zv/zt/zs(nx,ny,nz-1) REAL(4) (levels 1..nz-1 of one time record; level nz is never read,
 *       src/cdfmoc.f90:355), dmoc(nb,ny,nz) REAL(8) (cdfmoc.f90:287), dmoc(nb,nbins,ny) REAL(8) (cdfmocsig.f90:313).
 *   - The caller owns all host memory.  setup copies mesh/mask fields to the device (resident until teardown).
 *     A buffer given to *_submit must stay untouched until the matching *_fetch returns.  Host buffers from
 *     cdfgpu_pinned_alloc() make the H2D copy asynchronous (side stream, overlaps the previous record's kernel);
 *     pageable memory works but the copy is then staged by the driver.
 *   - One process drives one GPU (cdfgpu_init(device)) or several (cdfgpu_init_multi / $CDFGPU_DEVICES: records or
 *     latitude bands are distributed behind this ABI, results come back device -> host).  The one-process-per-GPU
 *     deployment (torchrun) distributes records or bands in the host layer (pass the band's rows, see j_first_global)
 *     and gathers the per-rank slabs there over NCCL.  Either way the path has no data-path collective.
 *   - Not re-entrant: call from one host thread (the reference's call sites are single-threaded).
 *   - There is NO CPU fallback: without a usable CUDA device every call fails with CDFGPU_ERR_NODEVICE.
 */
#ifndef CDFGPU_H
#define CDFGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CDFGPU_OK 0
#define CDFGPU_ERR_CUDA 1     /* a CUDA runtime call failed; see cdfgpu_last_error() */
#define CDFGPU_ERR_ARG 2      /* invalid argument */
#define CDFGPU_ERR_STATE 3    /* call order violated (no init / no setup / slot never submitted) */
#define CDFGPU_ERR_NOMEM 4    /* device or pinned allocation failed */
#define CDFGPU_ERR_NODEVICE 5 /* no CUDA device / driver */

#define CDFGPU_EOS_EOS80 0   /* polynomial EOS-80  (eos_init default,  src/eos.f90:408-466) */
#define CDFGPU_EOS_TEOS10 1  /* polynomial TEOS-10 (-teos10,           src/eos.f90:221-279) */
#define CDFGPU_EOS_NEUTRAL 2 /* neutral density    (-ntr, sigmantr,    src/eos.f90:661-684) */

#define CDFGPU_MAX_SLOTS 8
#define CDFGPU_MAX_BASINS 8

/* ---- lifecycle ------------------------------------------------------------------------------------------- */
/* Select the CUDA device (device < 0: $CDFGPU_DEVICE, else 0), create the compute and copy streams.
 * nslots (1..CDFGPU_MAX_SLOTS, 0 = default 3) is the depth of the record pipeline. */
int cdfgpu_init(int device, int nslots);
/* ONE host process, SEVERAL devices (the reference's host is a single process looping over the records, src/cdfmoc.f90:338,
 * src/cdfmocsig.f90:361).  cdfgpu_init(-1, n) honours $CDFGPU_DEVICES = N and $CDFGPU_SHARD = time | lat; cdfgpu_init_multi
 * asks for it explicitly (ndev = 0: $CDFGPU_DEVICES; shard 0 = time, 1 = lat).  Devices are $CDFGPU_DEVICE .. +N-1.
 *   time: slot s runs on device s mod N -- each device has its own record pipeline of `nslots` slots, so the host may keep
 *         cdfgpu_nslots() = N * nslots records in flight (submit slot jt mod cdfgpu_nslots(), fetch in the same order);
 *   lat : every record is split into N latitude bands: *_submit scatters them, *_fetch assembles the slab on the host.
 * cdfmoc / cdfmocsig setup, set_e3v, submit, fetch, kernel_ms, -isodep work under both; cdfmoc -decomp and the cdfmaxmoc
 * epilogue under time sharding only; the entry points that take device pointers (*_compute_device, *_device) need a single device.  Results are
 * bit-identical to a single device.  The cdfzonal and cdfmhst record pipelines (*_submit / *_fetch) are time-sharded the
 * same way (their synchronous calls on the first device), cdftransig runs on the first device; under lat every record and
 * plan of cdfzonal, cdfmhst and cdftransig is split into min(N, ny) latitude bands, synchronous calls included.  cdfsigtrp
 * runs on the first device. */
int cdfgpu_init_multi(int ndev, int shard, int nslots);
int cdfgpu_warmup(void);      /* create the CUDA contexts cdfgpu_init(-1, .) will use; callable from a helper thread at start-up */
int cdfgpu_num_devices(void); /* devices this process drives (0 before cdfgpu_init) */
int cdfgpu_nslots(void);      /* record slots the host may keep in flight */
int cdfgpu_finalize(void);
int cdfgpu_synchronize(void);
const char *cdfgpu_strerror(int code);
const char *cdfgpu_last_error(void);
int cdfgpu_device_count(void); /* >= 0, or -CDFGPU_ERR_* */
int cdfgpu_abi_version(void);
/* Page-locked host buffers for NF90_GET_VAR to fill (Fortran: c_f_pointer onto the returned address). */
void *cdfgpu_pinned_alloc(size_t nbytes);
int cdfgpu_pinned_free(void *p);
/* Ceiling of the record pipeline's input leg on this platform: GB/s of `reps` asynchronous copies of a pinned host buffer
 * to the device on the library's copy stream, with nothing else running. */
int cdfgpu_h2d_probe(const void *pinned, size_t nbytes, int reps, double *gbs);
/* Number of kernels this library has launched since cdfgpu_init (bench.py's gpu_launches). */
unsigned long long cdfgpu_launch_count(void);
/* K3: records handed to *_submit are RAW big-endian NetCDF-3 bytes (what fread delivers; the XDR decode libnetcdf
 * does on the CPU inside NF90_GET_VAR, src/cdfio.F90:1593): the byte swap then runs on the device, fused in front of
 * the record's kernel.  on = 0 (default): host-endian REAL(4) as NF90_GET_VAR returns them.  The flag is process-wide: it
 * applies to every device, and cdfgpu_finalize resets it to 0. */
int cdfgpu_set_input_big_endian(int on);
/* K3b: 16-bit packed records (NC_SHORT with scale_factor / add_offset, as cdf16bit writes them) unpacked on the device.
 * field is the position of the array in the submit calls: 0 = zv, 1 = zt, 2 = zs, 3 = zveiv, 4 = e3v_vvl.  With
 * CDFGPU_INPUT_I16, the `const float *` that cdfmoc_gpu_submit, cdfmoc_gpu_decomp_submit (fields 0-2) and
 * cdfmocsig_gpu_submit take for that field points at nx*ny*(nz-1) INTEGER(2) values instead (what NF90_GET_VAR into an
 * INTEGER(2) array delivers, or the raw file bytes when cdfgpu_set_input_big_endian is on: the 16-bit swap then runs in the
 * unpack kernel, and the field gets no 32-bit swap).  The device applies what getvar applies (src/cdfio.F90:1599-1605), bit
 * for bit: x = value; x = x*scale_factor where x /= spval (if scale_factor /= 1); x = x+add_offset where x /= spval (if
 * add_offset /= 0).  savelog10 is not offered.  CDFGPU_INPUT_F32 (the default) resets the field to REAL(4).  The setting
 * applies to every device of the process and lasts until changed, across cdfgpu_finalize; the *_compute_device entry
 * points are not affected.
 * CDFGPU_ERR_ARG for a field outside 0..4, an unknown type, or a non-finite scale_factor / add_offset. */
#define CDFGPU_INPUT_F32 0 /* REAL(4) as today (default) */
#define CDFGPU_INPUT_I16 1 /* NC_SHORT: decoded on the device as getvar does (cdfio.F90:1599-1605) */
int cdfgpu_set_input_packing(int field, int type, float scale_factor, float add_offset, float spval);
/* The same K3 / K3b input path for the synchronous sibling calls: how the record arrays of one call are stored.
 *   call = CDFGPU_CALL_ZONAL   (cdfzonal_gpu_sum / _mean: field 0 zv),
 *          CDFGPU_CALL_MHST    (cdfmhst_gpu_record: 0 zvt, 1 zvs),
 *          CDFGPU_CALL_MHST_VTS (cdfmhst_gpu_record_vts: 0 zv, 1 zt, 2 zs),
 *          CDFGPU_CALL_TRANSIG (cdftransig_gpu_record: 0 zu, 1 zv, 2 zt, 3 zs, 4 e3u_vvl, 5 e3v_vvl).
 *   type CDFGPU_INPUT_F32 | CDFGPU_INPUT_I16 with scale_factor / add_offset / spval as for cdfgpu_set_input_packing (the
 *   array then holds as many INTEGER(2) values as the call reads REAL(4) values); big_endian = 1: the array holds the raw
 *   file bytes (K3 swap, or the 16-bit swap of K3b).  A field never declared is host-order REAL(4).
 * The zonal and mhst calls do not look at cdfgpu_set_input_big_endian; cdftransig_gpu_record swaps a field when it is declared
 * big-endian OR that process-wide flag is on.  Independent of cdfgpu_set_input_packing (the submit fields).  Process-wide,
 * until changed, across cdfgpu_finalize.  CDFGPU_ERR_ARG for an unknown call, a field outside the call's list, an unknown type, or a non-finite
 * scale_factor / add_offset with CDFGPU_INPUT_I16. */
#define CDFGPU_CALL_ZONAL 0
#define CDFGPU_CALL_MHST 1
#define CDFGPU_CALL_MHST_VTS 2
#define CDFGPU_CALL_TRANSIG 3
int cdfgpu_set_sibling_input(int call, int field, int type, int big_endian, float scale_factor, float add_offset, float spval);
/* *_compute_device on a CALLER's stream: consecutive K1 / K2 launches overlap (programmatic dependent launch), and a launch
 * may read its device inputs before its predecessor on that stream has finished.  That is only safe when the inputs were
 * complete before the predecessor was enqueued (resident records).  on = 0 (default): every launch on a caller stream waits
 * for its predecessor before its first load (safe when a caller kernel right in front produces the inputs); on = 1: the
 * caller guarantees resident, synchronised inputs and gets the overlap.  Launches on the library's own streams are ordered
 * by the library itself.  The flag is process-wide, and cdfgpu_finalize resets it to 0. */
int cdfgpu_set_device_inputs_ready(int on);
/* Instruction-issue ceilings of the device, measured (the second bound of K2 beside HBM, bench.py): kind 0 = DFMA, 1 = FFMA,
 * 2 = FFMA2 (packed fp32), 3 = integer, 4 = FFMA and integer alternating.  out3 = { warp-instructions per clock and SM,
 * 1e9 warp-instructions per second over the chip, SM clock (MHz) during the run }. */
int cdfgpu_microbench(int kind, double *out3);

/* ---- cdfmoc: depth-space MOC ------------------------------------------------------------------------------
 * setup   replaces the one-time part of src/cdfmoc.f90:306,325-336,343-348:
 *           e1v     (nx,ny)      cdfmoc.f90:306
 *           e3v     (nx,ny,nz)   ALREADY multiplied by vmask(k) as get_e3v does (cdfmoc.f90:590-594)
 *           ibmask  (nb,nx,ny)   assembled as cdfmoc.f90:325-336 (global i=1,nx already zeroed)
 * set_e3v replaces the per-record reload under -vvl (cdfmoc.f90:339-348).
 * submit  enqueues record jt: H2D of zv on the copy stream, then the fused zonal-integral + scan kernel.
 * fetch   blocks until the slot's record is done and writes dmoc(nb,ny,nz) in Sv, already integrated from the
 *         bottom (cdfmoc.f90:382-388); dmoc(:,:,nz) = 0.
 * compute_device: same kernel on a record that is already in device memory (d_zv, d_dmoc device pointers,
 *         `stream` a cudaStream_t or NULL for the library's compute stream); asynchronous.  All compute_device calls on
 *         caller streams share one set of scheduling counters: issue them on ONE stream (or order the streams yourself).
 * Consecutive cdfmoc (and cdfmocsig) kernels of one stream are launched with programmatic stream serialization: the
 * next one may start while the previous one drains, but stores nothing before its predecessor is complete, so stream
 * order holds for every consumer (copies, events, kernels launched the ordinary way), and two launches may share an
 * output slab.  $CDFGPU_K1_PDL=0 / $CDFGPU_K2_PDL=0 restore plain launches.
 * Limit: the kernel keeps 8 x (nz-1) x nb fp64 column sums per block in shared memory; setup refuses with CDFGPU_ERR_ARG
 * (before any launch, the previous plan left as it was) when that exceeds the device's opt-in shared memory per block
 * (227 KB on a B200: nb = 8 up to nz = 455, nb = 5 up to nz = 727). */
int cdfmoc_gpu_setup(int nx, int ny, int nz, int nb, const float *e1v, const float *e3v, const int16_t *ibmask);
int cdfmoc_gpu_set_e3v(const float *e3v);
int cdfmoc_gpu_submit(int slot, int jt, const float *zv);
int cdfmoc_gpu_fetch(int slot, double *dmoc);
int cdfmoc_gpu_compute_device(const float *d_zv, double *d_dmoc, void *stream);
/* The same over nrec device-resident records in ONE launch (d_zv, d_dmoc: HOST arrays of nrec device pointers): the
 * work units run over (record, row, levels), so launch overhead, ramp-up and tail are paid once per batch. */
int cdfmoc_gpu_compute_device_batch(const float *const *d_zv, double *const *d_dmoc, int nrec, void *stream);
int cdfmoc_gpu_kernel_ms(int slot, float *ms); /* device time of the slot's last kernel, CUDA events */
/* Optional epilogue on the slot's streamfunction slab: the window extrema cdfmaxmoc computes from moc.nc
 * (src/cdfmaxmoc.f90:158-167).  Values are taken as REAL(4) (what the file holds); window bounds are 1-based
 * inclusive indices as found by cdfmaxmoc.f90:145-155; MAXLOC/MINLOC tie rule = first in (j fastest, k) order.
 * Non-finite values follow gfortran's MAXVAL/MAXLOC: NaN cells are skipped; a window of NaN cells only gives NaN
 * extrema located at its first cell (ijmin, ikmin); a window of -Inf cells (max) or +Inf cells (min) gives that
 * infinity at its first cell.  The sign of a zero extremum is that of the first cell holding it.
 * ovt[0..1] = max, min (Sv); loc[0..3] = jj of max, jk of max, jj of min, jk of min (1-based). */
int cdfmoc_gpu_maxmoc(int slot, int basin, int ijmin, int ijmax, int ikmin, int ikmax, float *ovt, int *loc);
/* -decomp (src/cdfmoc.f90:290-304,353,360-365,390-517): barotropic / geostrophic-shear / ageostrophic split.
 * decomp_setup (after cdfmoc_gpu_setup): e1u, gphiv (nx,ny); gdept (nz); umask, tmask (nx,ny,nz-1 levels used) as the
 *   INTEGER(2) planes the reference reads level by level (:439-440); teos10 selects the EOS of sigmai (:443).
 * decomp_submit: one record of V, T, S (nx,ny,nz-1); computes the total MOC and the three components.
 *   ONE decomposition is in flight per device: the component slabs are plan-wide, so a decomp_submit on another slot
 *   before the pending one is fetched (and a decomp_fetch of any other slot) fails with CDFGPU_ERR_STATE.
 * decomp_fetch : dmoc, dmoc_sh, dmoc_bt, dmoc_ag, each (nb,ny,nz) in Sv.  dmoc_sh starts from zero for every record
 *   (the reference never initialises it, cdfmoc.f90:299,471, which is only meaningful for a single record). */
int cdfmoc_gpu_decomp_setup(int teos10, const float *e1u, const float *gphiv, const float *gdept, const int16_t *umask,
                            const int16_t *tmask);
int cdfmoc_gpu_decomp_submit(int slot, int jt, const float *zv, const float *zt, const float *zs);
int cdfmoc_gpu_decomp_fetch(int slot, double *dmoc, double *dmoc_sh, double *dmoc_bt, double *dmoc_ag);
/* Device-resident records (the *_device rules above cdfzonal_gpu_sum_device apply: enqueue only, stream NULL = the library's
 * compute stream, inputs may come from the kernel right before the call, cdfgpu_set_device_inputs_ready as for
 * compute_device, 16-byte aligned pointers, one device only, CDFGPU_ERR_NODEVICE without a device).  Caller-stream calls
 * share compute_device's scheduling counters: issue them on ONE stream.  Whatever rewrites or frees data these calls read
 * (setup, set_e3v, decomp_setup, maxmoc_windows, teardown) first waits for the device once a device call has been made.
 * decomp_device: -decomp on device-resident V, T, S (nx,ny,nz-1); outputs (nb,ny,nz) fp64 on the device, Sv, as
 *   decomp_fetch gives them.  It takes no pipeline slot and may run beside records in flight; its working fields are the
 *   plan's, so decompositions on different streams take turns. */
int cdfmoc_gpu_decomp_device(const float *d_zv, const float *d_zt, const float *d_zs, double *d_dmoc,
                             double *d_dmoc_sh, double *d_dmoc_bt, double *d_dmoc_ag, void *stream);
/* cdfmaxmoc over a device slab: the run's windows once (host array win(5,nwin): basin 0-based as cdfmoc_gpu_maxmoc, ijmin,
 * ijmax, ikmin, ikmax 1-based inclusive; checked against the current plan, CDFGPU_ERR_ARG otherwise), then every window of
 * a device slab (nb,ny,nz) in ONE launch: ovt(2,nwin) = max, min; loc(4,nwin) = jj max, jk max, jj min, jk min (1-based),
 * with cdfmoc_gpu_maxmoc's rules.  maxmoc_device fails with CDFGPU_ERR_STATE before any windows are set and after a
 * cdfmoc_gpu_setup (which drops them). */
int cdfmoc_gpu_maxmoc_windows(int nwin, const int32_t *win);
int cdfmoc_gpu_maxmoc_device(const double *d_dmoc, float *d_ovt, int32_t *d_loc, void *stream);
int cdfmoc_gpu_teardown(void);

/* ---- cdfmocsig: density-space MOC -------------------------------------------------------------------------
 * setup   replaces src/cdfmocsig.f90:325,347-359 and fixes the binning (cdfmocsig.f90:265-304):
 *           e3v (nx,ny,nz) is the UNmasked e3v of mesh_zgr (cdfmocsig.f90:388; pass e31d(k) planes for -full),
 *           or NULL when every submit brings its own (-vvl).
 *           zspv/zspt/zsps: missing values of V, T, S (getspval, cdfmocsig.f90:227-229).
 *           eos: CDFGPU_EOS_*; pref: -r value (ignored for NEUTRAL).
 *           j_first_global / ny_global: when the caller hands over a latitude band, the 0-based global index of
 *           the band's first row and the global row count, so that the reference's skipping of the first and
 *           last global row (cdfmocsig.f90:405-407) is reproduced; pass 0 and ny for the whole domain.
 * submit  enqueues record jt: raw file values of zv, zt, zs (nx,ny,nz-1); the missing-value scrub
 *           (cdfmocsig.f90:375,383-384), optional bolus velocity (zveiv, -eiv, :376-379), area, EOS, bin and
 *           scatter-add are fused in one kernel.
 * fetch   dmoc(nb,nbins,ny) in Sv, integrated from the densest bin (cdfmocsig.f90:471-475).
 * bins_device: diagnostic for parity tests -- the bin index (1..nbins) of every cell of a device-resident
 *           record, computed by the same device function the fused kernel uses. */
int cdfmocsig_gpu_setup(int nx, int ny, int nz, int nb, int nbins, float sigmin, float sigstp, float pref, int eos,
                        const float *e1v, const float *e3v, const int16_t *ibmask, float zspv, float zspt, float zsps,
                        int j_first_global, int ny_global);
int cdfmocsig_gpu_submit(int slot, int jt, const float *zv, const float *zt, const float *zs, const float *zveiv,
                         const float *e3v_vvl);
int cdfmocsig_gpu_fetch(int slot, double *dmoc);
/* -isodep (src/cdfmocsig.f90:319-322,423-430,444-454,463-469): zonal mean of the isopycnal depths.
 * set_isodep(gdept(nz)) after setup enables it for the following submits (NULL switches it off); fetch_isodep gives
 * depi(nb,nbins,ny) in metres (negative down, as the reference's gdep = -gdept), 99999. where a class is empty.
 * When the three histograms of -isodep (3 x nbins x distinct basin-mask combinations doubles) do not fit in one CTA's
 * shared memory, set_isodep returns CDFGPU_ERR_ARG and leaves -isodep off; the plan keeps working without it. */
int cdfmocsig_gpu_set_isodep(const float *gdept);
int cdfmocsig_gpu_fetch_isodep(int slot, double *depi);
int cdfmocsig_gpu_compute_device(const float *d_zv, const float *d_zt, const float *d_zs, const float *d_zveiv,
                                 const float *d_e3v_vvl, double *d_dmoc, void *stream);
/* -isodep on device-resident records: dmoc as cdfmocsig_gpu_compute_device, depi (nb,nbins,ny) as fetch_isodep, both device
 * pointers.  CDFGPU_ERR_STATE unless cdfmocsig_gpu_set_isodep has enabled -isodep; otherwise the *_device rules above
 * cdfzonal_gpu_sum_device apply (16-byte aligned pointers, one device, CDFGPU_ERR_NODEVICE without a device). */
int cdfmocsig_gpu_compute_device_isodep(const float *d_zv, const float *d_zt, const float *d_zs, const float *d_zveiv,
                                        const float *d_e3v_vvl, double *d_dmoc, double *d_depi, void *stream);
int cdfmocsig_gpu_bins_device(const float *d_zt, const float *d_zs, int32_t *d_ibin, void *stream);
/* The same, plus how the three tiers of the bin function shared the work (host array): stats3[0] = cells evaluated,
 * [1] = cells the fp32 tier did not accept, [2] = cells that took the reference chain.  Blocks until done. */
int cdfmocsig_gpu_bins_device_stats(const float *d_zt, const float *d_zs, int32_t *d_ibin, unsigned long long *stats3,
                                    void *stream);
/* Diagnostics of the current plan: info8 = { fp32 tier on, fp64-FMA tier on, bound on |sigma_fp32 - sigma_reference| (kg/m3),
 * fp32 margin (bin units), fp64 margin (bin units), chunks of levels per row, levels per chunk, resident CTAs (0 before
 * the first launch) }. */
int cdfmocsig_gpu_filter_info(double *info8);
int cdfmocsig_gpu_kernel_ms(int slot, float *ms);
int cdfmocsig_gpu_teardown(void);

/* ---- sibling tools: the same masked zonal integral behind other command lines (SURVEY.md section 8 f3) --------------
 * Synchronous entry points on host buffers (pinned or pageable); one plan per tool and process (replayed on every device
 * under time sharding).
 *
 * Record pipelines, the way of cdfmoc_gpu_submit / _fetch: a submit copies its record on the copy stream once the slot's
 * previous kernel has read its inputs, and enqueues the decode (cdfgpu_set_sibling_input) and the kernel on the compute
 * stream, then returns; the matching fetch copies the result back and blocks.  The host reads record n+1 while record n
 * crosses PCIe.
 *   - slots 0 .. cdfgpu_nslots()-1.  Under time sharding slot s runs on device s mod N (local slot s / N); under latitude
 *     sharding every band device holds its share of every slot.  Fetch in any order; one record per slot at a time
 *     (a submit on a slot whose record has not been fetched: CDFGPU_ERR_STATE).
 *   - A host buffer given to a submit stays untouched until the matching fetch returns.
 *   - The field declarations (cdfgpu_set_sibling_input) are read at submit: a record in flight keeps the decoding it was
 *     submitted with.
 *   - The synchronous calls are submit on slot 0 and fetch; they fail with CDFGPU_ERR_STATE while a record of the same
 *     tool is in flight.  Setup and teardown wait for the records in flight and drop their results: a fetch afterwards
 *     fails with CDFGPU_ERR_STATE, as does a fetch of a slot with nothing submitted.  A slot out of range: CDFGPU_ERR_ARG.
 *   - Per-slot device buffers are allocated on a slot's first submit (slot 0's by setup).
 *   - *_kernel_ms reports the record of the last fetch.
 *
 * cdfzonalsum / cdfzonalmean -- replace the loop nests src/cdfzonalsum.f90:309-322 and src/cdfzonalmean.f90:312-344.
 *   setup: e1, e2 (nx,ny) horizontal metrics of the variable's C-grid point (dl_surf = 1.d0*e1*e2, cdfzonalsum.f90:257);
 *          zmask (nb,nx,ny) REAL(4) basin masks as assembled at cdfzonalsum.f90:286-296 (basin fastest);
 *          zmaskvar (nx,ny,nk) the variable's mask, every level (read level by level at :306).
 *   sum  : one 3-D record zv (nx,ny,nk) -> dzosum(ny,nk,nb) REAL(8) = SUM_i dl_surf*dble(zmask*zmaskvar*zv) / alpha(j)
 *          (alpha (ny) REAL(4), the -pdeg normalisation of :260-265; NULL = 1).
 *   mean : dzomean(ny,nk,nb) = SUM_i dl_surf*dtmp / SUM_i dl_surf*zmask*zmaskvar, zspval where the area is zero; with
 *          lmax the zonal maximum and non-zero minimum of dtmp, rzomax / rzomin (ny,nk,nb) REAL(4) (:325-326,339-342).
 *          A NaN dtmp never changes rzomax / rzomin: a row whose every dtmp is NaN keeps -1.e20 / 1.e20 (its mean is NaN). */
int cdfzonal_gpu_setup(int nx, int ny, int nk, int nb, const float *e1, const float *e2, const float *zmask,
                       const float *zmaskvar);
int cdfzonal_gpu_sum(const float *zv, const float *alpha, double *dzosum);
int cdfzonal_gpu_mean(const float *zv, float zspval, int lmax, double *dzomean, float *rzomax, float *rzomin);
/* pipeline: the same record as cdfzonal_gpu_sum / _mean on a slot; fetch writes dzo (dzosum or dzomean), and rzomax /
 * rzomin only when the submit was a mean with lmax (they may be NULL otherwise) */
int cdfzonal_gpu_submit_sum(int slot, const float *zv, const float *alpha);
int cdfzonal_gpu_submit_mean(int slot, const float *zv, float zspval, int lmax);
int cdfzonal_gpu_fetch(int slot, double *dzo, float *rzomax, float *rzomin);
int cdfzonal_gpu_kernel_ms(float *ms); /* device time of the last sum / mean kernel */
int cdfzonal_gpu_teardown(void);
/* Device-resident records (the *_device entry points of cdfzonal, cdfmhst and cdftransig): the same shapes, layouts and
 * values as the host-array call beside them, but every array is a DEVICE pointer and what that call writes to the host goes
 * to the caller's device buffer.
 *   - stream: a cudaStream_t, or NULL for the library's compute stream.  A call only enqueues work: it never synchronises the
 *     host and makes no host <-> device copy.  A result is complete once the stream reaches the point after the call; the
 *     inputs may come from the kernel right before the call on the same stream.  (cdftransig_gpu_record_device waits for the
 *     device once when another plan has loaded the other EOS coefficient set since, as cdfmocsig_gpu_compute_device does.)
 *   - Inputs are host-order REAL(4): the declarations of cdfgpu_set_sibling_input apply to host arrays only.
 *   - Every pointer must be 16-byte aligned (K4 / K5 issue 16-byte loads and derive a row's misalignment from its element
 *     index).  cudaMalloc and torch allocations are; a view at an odd offset is not: CDFGPU_ERR_ARG.
 *   - One device only: with several (cdfgpu_init_multi / $CDFGPU_DEVICES) CDFGPU_ERR_STATE.
 *   - CDFGPU_ERR_STATE before setup, CDFGPU_ERR_ARG for a null required pointer, CDFGPU_ERR_NODEVICE without any device.
 *   - The cdfzonal and cdfmhst device calls use no pipeline slot: they may run beside records in flight (they share only the
 *     read-only plan).  _vts keeps its V-point products in one plan buffer (allocated on its first call); calls on
 *     different streams take turns on it.  Teardown and setup wait for every device call made so far. */
int cdfzonal_gpu_sum_device(const float *d_zv, const float *d_alpha, double *d_dzosum, void *stream); /* d_alpha NULL = 1 */
int cdfzonal_gpu_mean_device(const float *d_zv, float zspval, int lmax, double *d_dzomean, float *d_rzomax, float *d_rzomin,
                             void *stream);
/* cdfmhst (-vt file mode) -- replaces src/cdfmhst.f90:303-366: vertical integral of vomevt / vomevs * e1v * e3v (heat
 * scaled by pprau0*pprcp) followed by the masked zonal sums.
 *   setup : e1v (nx,ny); e3v (nx,ny,nz) as read from the mesh file (or e31d(k) planes with -full); vmask1 = vmask(k=1);
 *           atl, pac, ind (nx,ny) REAL(4) basin masks, or all three NULL when there is no basin file.
 *   record: zvt, zvs (nx,ny,nz) -> heat, salt (ny,4,nlev) REAL(8): the raw sums dzonal_heat_* / dzonal_salt_* in the order
 *           glo, atl, pac, ind (glo over i = 2..npiglo-1, :341-344); nlev = nz with zdim (the sums after every level,
 *           :375) else 1 (after the last level).  The caller forms inp = ind + pac, inp0 = glo - atl, divides by 1.d15 /
 *           1.d6 and replaces zeros by ppspval (:384-441). */
int cdfmhst_gpu_setup(int nx, int ny, int nz, const float *e1v, const float *e3v, const float *vmask1, const float *atl,
                      const float *pac, const float *ind);
int cdfmhst_gpu_record(const float *zvt, const float *zvs, int zdim, double *heat, double *salt);
/* cdfmhst -v/-t[-s] mode (src/cdfmhst.f90:313-323): zv, zt, zs (nx,ny,nz) as read; the device forms
 * zvt = fl32(fl32(0.5*fl32(zt(j)+zt(j+1)))*zv), zvs likewise, row npjglo = 0, then proceeds as cdfmhst_gpu_record. */
int cdfmhst_gpu_record_vts(const float *zv, const float *zt, const float *zs, int zdim, double *heat, double *salt);
/* pipeline: cdfmhst_gpu_record / _record_vts on a slot; fetch writes heat, salt as they do */
int cdfmhst_gpu_submit(int slot, const float *zvt, const float *zvs, int zdim);
int cdfmhst_gpu_submit_vts(int slot, const float *zv, const float *zt, const float *zs, int zdim);
int cdfmhst_gpu_fetch(int slot, double *heat, double *salt);
int cdfmhst_gpu_kernel_ms(float *ms);
int cdfmhst_gpu_teardown(void);
/* device-resident records, as cdfmhst_gpu_record / _record_vts (see the *_device rules above cdfzonal_gpu_sum_device) */
int cdfmhst_gpu_record_device(const float *d_zvt, const float *d_zvs, int zdim, double *d_heat, double *d_salt, void *stream);
int cdfmhst_gpu_record_vts_device(const float *d_zv, const float *d_zt, const float *d_zs, int zdim, double *d_heat, double *d_salt,
                                  void *stream);

/* cdftransig_xy3d -- replaces the frame body of src/cdftransig_xy3d.f90:396-461 (kernel K6): the volume transport of
 * every U / V cell accumulated in density classes, dusigsig / dvsigsig (nx,ny,nbins) REAL(8), resident on the device
 * across the frames of a run.
 *   setup : pref = -depref (sigma0 when 0), teos10; ds1min, ds1scalmin = MIN(ds1scalmin, ds1scal) (:213) and the
 *           step -> bin table itab(nsigmax) the caller builds as at :229-262 (1-based bins; a 0 skips the cell, where the
 *           reference would index dusigsig(:,:,0)); e2u, e1v (nx,ny); e3u, e3v (nx,ny,nz-1) (NULL with -vvl: then every
 *           record brings its own); lperio = the E-W periodicity test of :336.  Zeroes the accumulators.
 *   record: one time frame zu, zv, zt, zs (nx,ny,nz-1), all levels.  set_masks = 1 for the frames of the FIRST tag: the
 *           reference derives zmasku / zmaskv from those frames only (:410-415) and keeps the last for later tags.
 *   fetch : the raw sums; the caller divides by nframes and converts to REAL(4) (:466-473).
 *   submit: cdftransig_gpu_record as a pipeline on slot 0 .. nslots-1 of cdfgpu_init: the frames are accumulated in
 *           submission order, so the sums are bit-identical to the synchronous frame loop.  On the first device, or under
 *           latitude sharding on every device for its band of rows (each (i,j) column's sums stay on one device; per-device
 *           partial sums of whole frames would change their association, so time sharding does not spread the frames).
 *           The copy of a frame overlaps the previous frame's kernels; the field declarations are read at submit.
 *   wait  : blocks until the slot's host arrays have been copied to the device: they may be refilled.  fetch waits for
 *           every frame submitted.  wait of a slot with no frame pending, and cdftransig_gpu_record while a submitted
 *           frame has been neither waited for nor fetched: CDFGPU_ERR_STATE.  kernel_ms: the last frame submitted. */
int cdftransig_gpu_setup(int nx, int ny, int nz, int nbins, float pref, int teos10, double ds1min, double ds1scalmin,
                         int nsigmax, const int32_t *itab, const float *e2u, const float *e1v, const float *e3u,
                         const float *e3v, int lperio);
int cdftransig_gpu_record(const float *zu, const float *zv, const float *zt, const float *zs, const float *e3u_vvl,
                          const float *e3v_vvl, int set_masks);
int cdftransig_gpu_fetch(double *dusigsig, double *dvsigsig);
int cdftransig_gpu_submit(int slot, const float *zu, const float *zv, const float *zt, const float *zs, const float *e3u_vvl,
                          const float *e3v_vvl, int set_masks);
int cdftransig_gpu_wait(int slot);
int cdftransig_gpu_kernel_ms(float *ms); /* device time of the last record (both kernels) */
int cdftransig_gpu_teardown(void);
/* A device-resident frame, as cdftransig_gpu_record (see the *_device rules above cdfzonal_gpu_sum_device).  Frames of
 * _record, _submit and _record_device accumulate in CALL order into the one set of accumulators: a device frame waits for
 * the last library frame, and the next library submit, record, fetch or setup waits for the last device frame, so any mix
 * gives the sums of the all-host frame loop bit for bit.  d_e3u_vvl / d_e3v_vvl (required with -vvl) are read in place;
 * given to a fixed-e3 setup they apply to this frame only.
 * fetch_device: a device-to-device copy of the raw sums, after every frame so far; later frames wait for it. */
int cdftransig_gpu_record_device(const float *d_zu, const float *d_zv, const float *d_zt, const float *d_zs, const float *d_e3u_vvl,
                                 const float *d_e3v_vvl, int set_masks, void *stream);
int cdftransig_gpu_fetch_device(double *d_dusigsig, double *d_dvsigsig, void *stream);

/* cdfsigtrp -- replaces the compute part of one section, src/cdfsigtrp.f90:559-627 (kernel K7): density of the section,
 * depth of the nbins+1 class limits in every column, transport from the surface down to each of them, and the binned
 * transports.  The host program keeps reading its section slices and the preparation of :428-555; arrays are the
 * reference's own after that block, (npts,npk) Fortran order:
 *   eu (npts) e1v or e2u; de3 (npts,npk) REAL(4) values of the reference's REAL(8) de3; ddepu (npts,0:npk) REAL(8);
 *   gdepw (npk), or ddepw_brk (npts,npk) the column's own w depths with -brk (:608; then gdepw may be NULL);
 *   zu, zt, zs, zmask (npts,npk) after the missing-value scrub / averaging; nk the number of levels used (:449-454).
 *   mode 0: sigmai(zt,zs,refdep) (sigma0 when refdep = 0; teos10 selects the coefficient set), 1: sigmantr, 2: -temp.
 *   dsigma_min, dsigma_max, nbins: class limits dsigma_lev(1:nbins+1) as at :355-359.
 * Outputs (host, any but dtrpbin may be NULL): dsigma_lev (nbins+1); dsig (npts,0:nk); dhiso, dwtrp (npts,nbins+1);
 * dwtrpbin (npts,nbins); dtrpbin (nbins) = SUM over the section, in m3/s (the caller divides by 1.d6). */
int cdfsigtrp_gpu_section(int npts, int npk, int nk, const float *eu, const float *de3, const double *ddepu, const float *gdepw,
                          const float *ddepw_brk, const float *zu, const float *zt, const float *zs, const float *zmask, int mode,
                          float refdep, int teos10, double dsigma_min, double dsigma_max, int nbins, double *dsigma_lev,
                          double *dsig, double *dhiso, double *dwtrp, double *dwtrpbin, double *dtrpbin);
int cdfsigtrp_gpu_kernel_ms(float *ms); /* device time of the last section (four kernels) */
/* A list of sections cut from whole device-resident fields: the cutting and the preparation of :404-555 run on the device
 * too, and every section of the list goes through one batch of four launches (independent of nsec).  The result of every
 * section is bit-identical to cdfsigtrp_gpu_section on the slices the host would cut and prepare.
 * sections_setup: whole 3-D fields are (nx,ny,npk) REAL(4), Fortran order.
 *   ijbox (4,nsec): imin imax jmin jmax per section, 1-based F-point indices as in dens_section.dat.
 *     imin == imax: meridional, columns (imin, jmin+1..jmax), T/S averaged with imin+1, velocity U, metric e2u;
 *     jmin == jmax: zonal, columns (imin+1..imax, jmin), T/S averaged with jmin+1, velocity V, metric e1v read from
 *                   imin..imax-1 (one column before the data, as the reference reads it);
 *     neither, or no column: the section is skipped (npts_out 0, its dtrpbin row 0, its nk 0), as the twin skips it.
 *     A meridional section needs 1 <= imin, imin+1 <= nx, 0 <= jmin, jmax <= ny; a zonal one 1 <= imin, imax <= nx,
 *     1 <= jmin, jmin+1 <= ny: CDFGPU_ERR_ARG otherwise.
 *   e1v, e2u (nx,ny) (NULL when no section needs it); e3u, e3v, e3w (nx,ny,npk), or all three NULL with -full: then
 *   e3t_1d, e3w_1d (npk) are used.  A mesh array a section needs and does not get: CDFGPU_ERR_ARG.
 *   gdept_1d (npk) (only gdept(1) is read, for ddepu), gdepw (npk).  zspu, zspv, zsps: missing values of U, V, S.
 *   mode / refdep / teos10 / dsigma_min / dsigma_max / nbins as cdfsigtrp_gpu_section (the caller applies the -temp sign
 *   change); nsec <= 65535 and nbins <= 65534, else CDFGPU_ERR_ARG.  Out (host, either may be NULL): dsigma_lev (nbins+1),
 *   npts_out (nsec).  Replaces the previous plan.
 * sections_device: one record of U, V, T, S (nx,ny,npk) REAL(4) in device memory -> d_dtrpbin (nbins,nsec) REAL(8) in
 *   m3/s, d_nk (nsec) INTEGER (the levels used; NULL: not written).  d_zu3d may be NULL when no section is meridional,
 *   d_zv3d when none is zonal.  The *_device rules above cdfzonal_gpu_sum_device apply, except that pointers need only be
 *   aligned to their element: enqueue only, inputs may come from the kernel right before the call; one device only;
 *   CDFGPU_ERR_STATE before setup, CDFGPU_ERR_NODEVICE without any device.  The plan's scratch is shared: calls on
 *   different streams take turns on it.  mode 0 waits for the device once when another plan has loaded the other EOS
 *   coefficient set since.  cdfsigtrp_gpu_teardown (and setup, and cdfgpu_finalize) wait for every device call so far. */
int cdfsigtrp_gpu_sections_setup(int nx, int ny, int npk, int nsec, const int32_t *ijbox, const float *e1v, const float *e2u,
                                 const float *e3u, const float *e3v, const float *e3w, const float *e3t_1d, const float *e3w_1d,
                                 const float *gdept_1d, const float *gdepw, float zspu, float zspv, float zsps, int mode,
                                 float refdep, int teos10, double dsigma_min, double dsigma_max, int nbins,
                                 double *dsigma_lev, int32_t *npts_out);
int cdfsigtrp_gpu_sections_device(const float *d_zu3d, const float *d_zv3d, const float *d_zt3d, const float *d_zs3d,
                                  double *d_dtrpbin, int32_t *d_nk, void *stream);
int cdfsigtrp_gpu_teardown(void);

#ifdef __cplusplus
}
#endif
#endif /* CDFGPU_H */
