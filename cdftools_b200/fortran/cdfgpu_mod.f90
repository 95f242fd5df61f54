MODULE cdfgpu
  !!======================================================================
  !!                     ***  MODULE  cdfgpu  ***
  !! ISO_C_BINDING interface to libcdfgpu.so (include/cdfgpu.h): the B200
  !! implementation of the cdfmoc / cdfmocsig hot loops.
  !!
  !! This is the thin bind(C) layer a CDFTOOLS maintainer adds to src/ so that
  !!    src/cdfmoc.f90:352-388      ->  cdfmoc_gpu_submit / cdfmoc_gpu_fetch
  !!    src/cdfmocsig.f90:366-475   ->  cdfmocsig_gpu_submit / cdfmocsig_gpu_fetch
  !! The host program stays Fortran: same command line, same cdfio calls, same
  !! output file.  INTEGRATION.md shows the call-site patches.
  !!
  !! NOTE: gfortran / netcdf-fortran are not available in the build image of this
  !! repository, so this file is shipped as source and has NOT been compiled here.
  !! It only uses standard Fortran 2003 interoperability features.
  !!
  !! Array conventions: Fortran arrays are passed as they are declared in the
  !! reference (column-major), which is exactly the C [k][j][i] order the library
  !! expects -- no transposes:
  !!    e1v(npiglo,npjglo)  e3v(npiglo,npjglo,npk)  ibmask(nbasins,npiglo,npjglo)
  !!    zv(npiglo,npjglo,npk-1)   dmoc(nbasins,npjglo,npk) / dmoc(nvaro,nbins,npjglo)
  !!======================================================================
  USE, INTRINSIC :: ISO_C_BINDING
  IMPLICIT NONE
  PUBLIC

  INTEGER(C_INT), PARAMETER :: CDFGPU_OK = 0
  INTEGER(C_INT), PARAMETER :: CDFGPU_EOS_EOS80 = 0, CDFGPU_EOS_TEOS10 = 1, CDFGPU_EOS_NEUTRAL = 2
  INTEGER(C_INT), PARAMETER :: CDFGPU_INPUT_F32 = 0, CDFGPU_INPUT_I16 = 1
  INTEGER(C_INT), PARAMETER :: CDFGPU_CALL_ZONAL = 0, CDFGPU_CALL_MHST = 1, CDFGPU_CALL_MHST_VTS = 2, CDFGPU_CALL_TRANSIG = 3

  INTERFACE
     ! ---- lifecycle ---------------------------------------------------------
     INTEGER(C_INT) FUNCTION cdfgpu_init(device, nslots) BIND(C, NAME='cdfgpu_init')
       IMPORT :: C_INT
       INTEGER(C_INT), VALUE :: device, nslots
     END FUNCTION cdfgpu_init

     ! one host process, several devices: shard 0 = by time record (slot s on device MOD(s, ndev)), 1 = latitude bands;
     ! ndev = 0 reads $CDFGPU_DEVICES.  cdfgpu_init(-1, n) honours $CDFGPU_DEVICES / $CDFGPU_SHARD by itself.
     INTEGER(C_INT) FUNCTION cdfgpu_init_multi(ndev, shard, nslots) BIND(C, NAME='cdfgpu_init_multi')
       IMPORT :: C_INT
       INTEGER(C_INT), VALUE :: ndev, shard, nslots
     END FUNCTION cdfgpu_init_multi

     ! creates the CUDA contexts cdfgpu_init(-1, n) will use (callable from an OpenMP task at start-up, while the mesh is read)
     INTEGER(C_INT) FUNCTION cdfgpu_warmup() BIND(C, NAME='cdfgpu_warmup')
       IMPORT :: C_INT
     END FUNCTION cdfgpu_warmup

     INTEGER(C_INT) FUNCTION cdfgpu_num_devices() BIND(C, NAME='cdfgpu_num_devices')
       IMPORT :: C_INT
     END FUNCTION cdfgpu_num_devices

     ! record slots the host may keep in flight (ndev * nslots under time sharding): the DO jt loop submits record jt on
     ! slot MOD(jt-1, cdfgpu_nslots()) and fetches in the same order
     INTEGER(C_INT) FUNCTION cdfgpu_nslots() BIND(C, NAME='cdfgpu_nslots')
       IMPORT :: C_INT
     END FUNCTION cdfgpu_nslots

     INTEGER(C_INT) FUNCTION cdfgpu_finalize() BIND(C, NAME='cdfgpu_finalize')
       IMPORT :: C_INT
     END FUNCTION cdfgpu_finalize

     INTEGER(C_INT) FUNCTION cdfgpu_synchronize() BIND(C, NAME='cdfgpu_synchronize')
       IMPORT :: C_INT
     END FUNCTION cdfgpu_synchronize

     TYPE(C_PTR) FUNCTION cdfgpu_last_error() BIND(C, NAME='cdfgpu_last_error')
       IMPORT :: C_PTR
     END FUNCTION cdfgpu_last_error

     TYPE(C_PTR) FUNCTION cdfgpu_pinned_alloc(nbytes) BIND(C, NAME='cdfgpu_pinned_alloc')
       IMPORT :: C_PTR, C_SIZE_T
       INTEGER(C_SIZE_T), VALUE :: nbytes
     END FUNCTION cdfgpu_pinned_alloc

     INTEGER(C_INT) FUNCTION cdfgpu_pinned_free(p) BIND(C, NAME='cdfgpu_pinned_free')
       IMPORT :: C_INT, C_PTR
       TYPE(C_PTR), VALUE :: p
     END FUNCTION cdfgpu_pinned_free

     INTEGER(C_INT) FUNCTION cdfgpu_abi_version() BIND(C, NAME='cdfgpu_abi_version')
       IMPORT :: C_INT
     END FUNCTION cdfgpu_abi_version

     INTEGER(C_INT) FUNCTION cdfgpu_device_count() BIND(C, NAME='cdfgpu_device_count')
       IMPORT :: C_INT
     END FUNCTION cdfgpu_device_count

     ! device time (ms) of the last kernel of a slot / tool, for the timing prints of the host program
     INTEGER(C_INT) FUNCTION cdfmoc_gpu_kernel_ms(slot, ms) BIND(C, NAME='cdfmoc_gpu_kernel_ms')
       IMPORT :: C_INT, C_FLOAT
       INTEGER(C_INT), VALUE :: slot
       REAL(C_FLOAT), INTENT(out) :: ms
     END FUNCTION cdfmoc_gpu_kernel_ms

     INTEGER(C_INT) FUNCTION cdfmocsig_gpu_kernel_ms(slot, ms) BIND(C, NAME='cdfmocsig_gpu_kernel_ms')
       IMPORT :: C_INT, C_FLOAT
       INTEGER(C_INT), VALUE :: slot
       REAL(C_FLOAT), INTENT(out) :: ms
     END FUNCTION cdfmocsig_gpu_kernel_ms

     INTEGER(C_INT) FUNCTION cdfzonal_gpu_kernel_ms(ms) BIND(C, NAME='cdfzonal_gpu_kernel_ms')
       IMPORT :: C_INT, C_FLOAT
       REAL(C_FLOAT), INTENT(out) :: ms
     END FUNCTION cdfzonal_gpu_kernel_ms

     INTEGER(C_INT) FUNCTION cdfmhst_gpu_kernel_ms(ms) BIND(C, NAME='cdfmhst_gpu_kernel_ms')
       IMPORT :: C_INT, C_FLOAT
       REAL(C_FLOAT), INTENT(out) :: ms
     END FUNCTION cdfmhst_gpu_kernel_ms

     INTEGER(C_INT) FUNCTION cdftransig_gpu_kernel_ms(ms) BIND(C, NAME='cdftransig_gpu_kernel_ms')
       IMPORT :: C_INT, C_FLOAT
       REAL(C_FLOAT), INTENT(out) :: ms
     END FUNCTION cdftransig_gpu_kernel_ms

     ! records given to *_submit are raw big-endian file bytes: byte swap on the device
     INTEGER(C_INT) FUNCTION cdfgpu_set_input_big_endian(on) BIND(C, NAME='cdfgpu_set_input_big_endian')
       IMPORT :: C_INT
       INTEGER(C_INT), VALUE :: on
     END FUNCTION cdfgpu_set_input_big_endian

     ! field kfield (0 zv, 1 zt, 2 zs, 3 zveiv, 4 e3v_vvl) of the submit calls is INTEGER(2) (ktype CDFGPU_INPUT_I16),
     ! unpacked on the device as getvar does, or REAL(4) (CDFGPU_INPUT_F32, the default)
     INTEGER(C_INT) FUNCTION cdfgpu_set_input_packing(kfield, ktype, psf, pao, pspval) BIND(C, NAME='cdfgpu_set_input_packing')
       IMPORT :: C_INT, C_FLOAT
       INTEGER(C_INT), VALUE :: kfield, ktype
       REAL(C_FLOAT),  VALUE :: psf, pao, pspval
     END FUNCTION cdfgpu_set_input_packing

     ! record array kfield of the sibling call kcall (CDFGPU_CALL_*; fields in the order of the call's arguments) is
     ! INTEGER(2) (CDFGPU_INPUT_I16, unpacked on the device) or REAL(4); kbig_endian = 1: raw file bytes
     INTEGER(C_INT) FUNCTION cdfgpu_set_sibling_input(kcall, kfield, ktype, kbig_endian, psf, pao, pspval) &
          &                                          BIND(C, NAME='cdfgpu_set_sibling_input')
       IMPORT :: C_INT, C_FLOAT
       INTEGER(C_INT), VALUE :: kcall, kfield, ktype, kbig_endian
       REAL(C_FLOAT),  VALUE :: psf, pao, pspval
     END FUNCTION cdfgpu_set_sibling_input

     ! diagnostics of the current cdfmocsig plan (tiers of the bin function, work units): info(8), see cdfgpu.h
     INTEGER(C_INT) FUNCTION cdfmocsig_gpu_filter_info(info8) BIND(C, NAME='cdfmocsig_gpu_filter_info')
       IMPORT :: C_INT, C_DOUBLE
       REAL(C_DOUBLE), INTENT(out) :: info8(8)
     END FUNCTION cdfmocsig_gpu_filter_info

     ! ---- cdfmoc ------------------------------------------------------------
     INTEGER(C_INT) FUNCTION cdfmoc_gpu_setup(nx, ny, nz, nb, e1v, e3v, ibmask) BIND(C, NAME='cdfmoc_gpu_setup')
       IMPORT :: C_INT, C_FLOAT, C_INT16_T
       INTEGER(C_INT), VALUE :: nx, ny, nz, nb
       REAL(C_FLOAT),      INTENT(in) :: e1v(*), e3v(*)      ! e3v already * vmask (cdfmoc.f90:590-594)
       INTEGER(C_INT16_T), INTENT(in) :: ibmask(*)           ! (nbasins,npiglo,npjglo), cdfmoc.f90:325-336
     END FUNCTION cdfmoc_gpu_setup

     INTEGER(C_INT) FUNCTION cdfmoc_gpu_set_e3v(e3v) BIND(C, NAME='cdfmoc_gpu_set_e3v')
       IMPORT :: C_INT, C_FLOAT
       REAL(C_FLOAT), INTENT(in) :: e3v(*)                   ! -vvl: per-record e3v * vmask
     END FUNCTION cdfmoc_gpu_set_e3v

     INTEGER(C_INT) FUNCTION cdfmoc_gpu_submit(slot, jt, zv) BIND(C, NAME='cdfmoc_gpu_submit')
       IMPORT :: C_INT, C_FLOAT
       INTEGER(C_INT), VALUE :: slot, jt
       REAL(C_FLOAT), INTENT(in) :: zv(*)                    ! (npiglo,npjglo,npk-1), pinned
     END FUNCTION cdfmoc_gpu_submit

     INTEGER(C_INT) FUNCTION cdfmoc_gpu_fetch(slot, dmoc) BIND(C, NAME='cdfmoc_gpu_fetch')
       IMPORT :: C_INT, C_DOUBLE
       INTEGER(C_INT), VALUE :: slot
       REAL(C_DOUBLE), INTENT(out) :: dmoc(*)                ! (nbasins,npjglo,npk), Sv, integrated
     END FUNCTION cdfmoc_gpu_fetch

     ! cdfmaxmoc window search on the slot's device slab (cdfmaxmoc.f90:158-167)
     INTEGER(C_INT) FUNCTION cdfmoc_gpu_maxmoc(slot, basin, ijmin, ijmax, ikmin, ikmax, ovt, loc) &
          &                                    BIND(C, NAME='cdfmoc_gpu_maxmoc')
       IMPORT :: C_INT, C_FLOAT
       INTEGER(C_INT), VALUE :: slot, basin, ijmin, ijmax, ikmin, ikmax    ! basin 0-based, window 1-based inclusive
       REAL(C_FLOAT),  INTENT(out) :: ovt(2)                 ! max, min (Sv)
       INTEGER(C_INT), INTENT(out) :: loc(4)                 ! jj,jk of max ; jj,jk of min (1-based)
     END FUNCTION cdfmoc_gpu_maxmoc

     ! -decomp (cdfmoc.f90:390-517)
     INTEGER(C_INT) FUNCTION cdfmoc_gpu_decomp_setup(teos10, e1u, gphiv, gdept, iumask, itmask) &
          &                                          BIND(C, NAME='cdfmoc_gpu_decomp_setup')
       IMPORT :: C_INT, C_FLOAT, C_INT16_T
       INTEGER(C_INT), VALUE :: teos10
       REAL(C_FLOAT),      INTENT(in) :: e1u(*), gphiv(*), gdept(*)
       INTEGER(C_INT16_T), INTENT(in) :: iumask(*), itmask(*)   ! (npiglo,npjglo,npk-1)
     END FUNCTION cdfmoc_gpu_decomp_setup

     INTEGER(C_INT) FUNCTION cdfmoc_gpu_decomp_submit(slot, jt, zv, zt, zs) BIND(C, NAME='cdfmoc_gpu_decomp_submit')
       IMPORT :: C_INT, C_FLOAT
       INTEGER(C_INT), VALUE :: slot, jt
       REAL(C_FLOAT), INTENT(in) :: zv(*), zt(*), zs(*)
     END FUNCTION cdfmoc_gpu_decomp_submit

     INTEGER(C_INT) FUNCTION cdfmoc_gpu_decomp_fetch(slot, dmoc, dmoc_sh, dmoc_bt, dmoc_ag) &
          &                                          BIND(C, NAME='cdfmoc_gpu_decomp_fetch')
       IMPORT :: C_INT, C_DOUBLE
       INTEGER(C_INT), VALUE :: slot
       REAL(C_DOUBLE), INTENT(out) :: dmoc(*), dmoc_sh(*), dmoc_bt(*), dmoc_ag(*)   ! each (nbasins,npjglo,npk)
     END FUNCTION cdfmoc_gpu_decomp_fetch

     ! device-resident records (OpenACC host_data use_device / CUDA Fortran device arrays), as cdfzonal_gpu_sum_device:
     ! every array argument is the C_LOC of a DEVICE array, 16-byte aligned; stream a cudaStream_t or C_NULL_PTR
     INTEGER(C_INT) FUNCTION cdfmoc_gpu_decomp_device(d_zv, d_zt, d_zs, d_dmoc, d_dmoc_sh, d_dmoc_bt, d_dmoc_ag, stream) &
          &                                           BIND(C, NAME='cdfmoc_gpu_decomp_device')
       IMPORT :: C_INT, C_PTR
       TYPE(C_PTR), VALUE :: d_zv, d_zt, d_zs                ! (npiglo,npjglo,npk-1) REAL(4)
       TYPE(C_PTR), VALUE :: d_dmoc, d_dmoc_sh, d_dmoc_bt, d_dmoc_ag   ! each (nbasins,npjglo,npk) REAL(8), Sv
       TYPE(C_PTR), VALUE :: stream
     END FUNCTION cdfmoc_gpu_decomp_device

     ! cdfmaxmoc windows for cdfmoc_gpu_maxmoc_device, once per run (a HOST array)
     INTEGER(C_INT) FUNCTION cdfmoc_gpu_maxmoc_windows(nwin, win) BIND(C, NAME='cdfmoc_gpu_maxmoc_windows')
       IMPORT :: C_INT, C_INT32_T
       INTEGER(C_INT), VALUE :: nwin
       INTEGER(C_INT32_T), INTENT(in) :: win(5,*)            ! basin (0-based), ijmin, ijmax, ikmin, ikmax (1-based)
     END FUNCTION cdfmoc_gpu_maxmoc_windows

     INTEGER(C_INT) FUNCTION cdfmoc_gpu_maxmoc_device(d_dmoc, d_ovt, d_loc, stream) BIND(C, NAME='cdfmoc_gpu_maxmoc_device')
       IMPORT :: C_INT, C_PTR
       TYPE(C_PTR), VALUE :: d_dmoc                          ! (nbasins,npjglo,npk) REAL(8)
       TYPE(C_PTR), VALUE :: d_ovt                           ! (2,nwin) REAL(4): max, min
       TYPE(C_PTR), VALUE :: d_loc                           ! (4,nwin) INTEGER(4): jj,jk of max ; jj,jk of min
       TYPE(C_PTR), VALUE :: stream
     END FUNCTION cdfmoc_gpu_maxmoc_device

     INTEGER(C_INT) FUNCTION cdfmoc_gpu_teardown() BIND(C, NAME='cdfmoc_gpu_teardown')
       IMPORT :: C_INT
     END FUNCTION cdfmoc_gpu_teardown

     ! ---- cdfmocsig ---------------------------------------------------------
     INTEGER(C_INT) FUNCTION cdfmocsig_gpu_setup(nx, ny, nz, nb, nbins, sigmin, sigstp, pref, eos, e1v, e3v, &
          &                                      ibmask, zspv, zspt, zsps, j_first_global, ny_global)         &
          &                                      BIND(C, NAME='cdfmocsig_gpu_setup')
       IMPORT :: C_INT, C_FLOAT, C_INT16_T, C_PTR
       INTEGER(C_INT), VALUE :: nx, ny, nz, nb, nbins, eos, j_first_global, ny_global
       REAL(C_FLOAT),  VALUE :: sigmin, sigstp, pref, zspv, zspt, zsps
       REAL(C_FLOAT),      INTENT(in) :: e1v(*)
       TYPE(C_PTR), VALUE             :: e3v                 ! C_LOC(e3v3d) (UNmasked), or C_NULL_PTR with -vvl
       INTEGER(C_INT16_T), INTENT(in) :: ibmask(*)
     END FUNCTION cdfmocsig_gpu_setup

     INTEGER(C_INT) FUNCTION cdfmocsig_gpu_submit(slot, jt, zv, zt, zs, zveiv, e3v_vvl) BIND(C, NAME='cdfmocsig_gpu_submit')
       IMPORT :: C_INT, C_FLOAT, C_PTR
       INTEGER(C_INT), VALUE :: slot, jt
       REAL(C_FLOAT), INTENT(in) :: zv(*), zt(*), zs(*)      ! raw file values, (npiglo,npjglo,npk-1), pinned
       TYPE(C_PTR), VALUE :: zveiv, e3v_vvl                  ! C_LOC(...) or C_NULL_PTR
     END FUNCTION cdfmocsig_gpu_submit

     INTEGER(C_INT) FUNCTION cdfmocsig_gpu_fetch(slot, dmoc) BIND(C, NAME='cdfmocsig_gpu_fetch')
       IMPORT :: C_INT, C_DOUBLE
       INTEGER(C_INT), VALUE :: slot
       REAL(C_DOUBLE), INTENT(out) :: dmoc(*)                ! (nbasins,nbins,npjglo), Sv, integrated
     END FUNCTION cdfmocsig_gpu_fetch

     ! -isodep (cdfmocsig.f90:423-469)
     INTEGER(C_INT) FUNCTION cdfmocsig_gpu_set_isodep(gdept) BIND(C, NAME='cdfmocsig_gpu_set_isodep')
       IMPORT :: C_INT, C_FLOAT
       REAL(C_FLOAT), INTENT(in) :: gdept(*)                 ! (npk), positive depths; the library uses -gdept
     END FUNCTION cdfmocsig_gpu_set_isodep

     INTEGER(C_INT) FUNCTION cdfmocsig_gpu_fetch_isodep(slot, depi) BIND(C, NAME='cdfmocsig_gpu_fetch_isodep')
       IMPORT :: C_INT, C_DOUBLE
       INTEGER(C_INT), VALUE :: slot
       REAL(C_DOUBLE), INTENT(out) :: depi(*)                ! (nbasins,nbins,npjglo)
     END FUNCTION cdfmocsig_gpu_fetch_isodep

     ! -isodep on device-resident records (device arrays as cdfmoc_gpu_decomp_device)
     INTEGER(C_INT) FUNCTION cdfmocsig_gpu_compute_device_isodep(d_zv, d_zt, d_zs, d_zveiv, d_e3v_vvl, d_dmoc, d_depi, &
          &                                                      stream) BIND(C, NAME='cdfmocsig_gpu_compute_device_isodep')
       IMPORT :: C_INT, C_PTR
       TYPE(C_PTR), VALUE :: d_zv, d_zt, d_zs                ! (npiglo,npjglo,npk-1) REAL(4)
       TYPE(C_PTR), VALUE :: d_zveiv, d_e3v_vvl              ! (npiglo,npjglo,npk-1) REAL(4), or C_NULL_PTR
       TYPE(C_PTR), VALUE :: d_dmoc, d_depi                  ! each (nbasins,nbins,npjglo) REAL(8)
       TYPE(C_PTR), VALUE :: stream
     END FUNCTION cdfmocsig_gpu_compute_device_isodep

     INTEGER(C_INT) FUNCTION cdfmocsig_gpu_teardown() BIND(C, NAME='cdfmocsig_gpu_teardown')
       IMPORT :: C_INT
     END FUNCTION cdfmocsig_gpu_teardown
     ! ---- sibling tools: cdfzonalsum / cdfzonalmean / cdfmhst (include/cdfgpu.h, SURVEY 8 f3) ----
     INTEGER(C_INT) FUNCTION cdfzonal_gpu_setup(nx, ny, nk, nb, e1, e2, zmask, zmaskvar) BIND(C, NAME='cdfzonal_gpu_setup')
       IMPORT :: C_INT, C_FLOAT
       INTEGER(C_INT), VALUE :: nx, ny, nk, nb
       REAL(C_FLOAT), INTENT(in) :: e1(*), e2(*)            ! (npiglo,npjglo) metrics of the variable's grid point
       REAL(C_FLOAT), INTENT(in) :: zmask(*)                ! (npbasins,npiglo,npjglo), cdfzonalsum.f90:286-296
       REAL(C_FLOAT), INTENT(in) :: zmaskvar(*)             ! (npiglo,npjglo,npk) mask of the variable, every level
     END FUNCTION cdfzonal_gpu_setup

     INTEGER(C_INT) FUNCTION cdfzonal_gpu_sum(zv, alpha, dzosum) BIND(C, NAME='cdfzonal_gpu_sum')
       IMPORT :: C_INT, C_FLOAT, C_DOUBLE, C_PTR
       REAL(C_FLOAT), INTENT(in) :: zv(*)                   ! (npiglo,npjglo,npk) one record of one variable
       TYPE(C_PTR), VALUE :: alpha                          ! C_LOC(alpha(npjglo)) with -pdeg, else C_NULL_PTR
       REAL(C_DOUBLE), INTENT(out) :: dzosum(*)             ! (npjglo,npk,npbasins)
     END FUNCTION cdfzonal_gpu_sum

     INTEGER(C_INT) FUNCTION cdfzonal_gpu_mean(zv, zspval, lmax, dzomean, rzomax, rzomin) BIND(C, NAME='cdfzonal_gpu_mean')
       IMPORT :: C_INT, C_FLOAT, C_DOUBLE, C_PTR
       REAL(C_FLOAT), INTENT(in) :: zv(*)
       REAL(C_FLOAT), VALUE :: zspval
       INTEGER(C_INT), VALUE :: lmax                        ! 1 with -max
       REAL(C_DOUBLE), INTENT(out) :: dzomean(*)            ! (npjglo,npk,npbasins)
       TYPE(C_PTR), VALUE :: rzomax, rzomin                 ! C_LOC of (npjglo,npk,npbasins) REAL(4), or C_NULL_PTR
     END FUNCTION cdfzonal_gpu_mean

     ! record pipeline: submit on slot 0 .. cdfgpu_nslots()-1, fetch blocks; zv (and alpha) untouched until the fetch returns
     INTEGER(C_INT) FUNCTION cdfzonal_gpu_submit_sum(slot, zv, alpha) BIND(C, NAME='cdfzonal_gpu_submit_sum')
       IMPORT :: C_INT, C_FLOAT, C_PTR
       INTEGER(C_INT), VALUE :: slot
       REAL(C_FLOAT), INTENT(in) :: zv(*)                   ! (npiglo,npjglo,npk), pinned
       TYPE(C_PTR), VALUE :: alpha                          ! C_LOC(alpha(npjglo)) with -pdeg, else C_NULL_PTR
     END FUNCTION cdfzonal_gpu_submit_sum

     INTEGER(C_INT) FUNCTION cdfzonal_gpu_submit_mean(slot, zv, zspval, lmax) BIND(C, NAME='cdfzonal_gpu_submit_mean')
       IMPORT :: C_INT, C_FLOAT
       INTEGER(C_INT), VALUE :: slot
       REAL(C_FLOAT), INTENT(in) :: zv(*)                   ! (npiglo,npjglo,npk), pinned
       REAL(C_FLOAT), VALUE :: zspval
       INTEGER(C_INT), VALUE :: lmax                        ! 1 with -max
     END FUNCTION cdfzonal_gpu_submit_mean

     INTEGER(C_INT) FUNCTION cdfzonal_gpu_fetch(slot, dzo, rzomax, rzomin) BIND(C, NAME='cdfzonal_gpu_fetch')
       IMPORT :: C_INT, C_DOUBLE, C_PTR
       INTEGER(C_INT), VALUE :: slot
       REAL(C_DOUBLE), INTENT(out) :: dzo(*)                ! dzosum or dzomean (npjglo,npk,npbasins)
       TYPE(C_PTR), VALUE :: rzomax, rzomin                 ! C_LOC of (npjglo,npk,npbasins) REAL(4) after a mean with lmax
     END FUNCTION cdfzonal_gpu_fetch

     INTEGER(C_INT) FUNCTION cdfzonal_gpu_teardown() BIND(C, NAME='cdfzonal_gpu_teardown')
       IMPORT :: C_INT
     END FUNCTION cdfzonal_gpu_teardown

     ! device-resident records (OpenACC host_data use_device / CUDA Fortran device arrays): every array argument is the
     ! C_LOC of a DEVICE array of the host call's shape, 16-byte aligned; stream a cudaStream_t or C_NULL_PTR (the library's).
     ! The calls only enqueue work: results are complete once the stream has passed them.
     INTEGER(C_INT) FUNCTION cdfzonal_gpu_sum_device(d_zv, d_alpha, d_dzosum, stream) BIND(C, NAME='cdfzonal_gpu_sum_device')
       IMPORT :: C_INT, C_PTR
       TYPE(C_PTR), VALUE :: d_zv                           ! (npiglo,npjglo,npk) REAL(4)
       TYPE(C_PTR), VALUE :: d_alpha                        ! (npjglo) REAL(4) with -pdeg, else C_NULL_PTR
       TYPE(C_PTR), VALUE :: d_dzosum                       ! (npjglo,npk,npbasins) REAL(8)
       TYPE(C_PTR), VALUE :: stream
     END FUNCTION cdfzonal_gpu_sum_device

     INTEGER(C_INT) FUNCTION cdfzonal_gpu_mean_device(d_zv, zspval, lmax, d_dzomean, d_rzomax, d_rzomin, stream) &
          &                                          BIND(C, NAME='cdfzonal_gpu_mean_device')
       IMPORT :: C_INT, C_FLOAT, C_PTR
       TYPE(C_PTR), VALUE :: d_zv                           ! (npiglo,npjglo,npk) REAL(4)
       REAL(C_FLOAT), VALUE :: zspval
       INTEGER(C_INT), VALUE :: lmax                        ! 1 with -max
       TYPE(C_PTR), VALUE :: d_dzomean                      ! (npjglo,npk,npbasins) REAL(8)
       TYPE(C_PTR), VALUE :: d_rzomax, d_rzomin             ! (npjglo,npk,npbasins) REAL(4) with lmax, else C_NULL_PTR
       TYPE(C_PTR), VALUE :: stream
     END FUNCTION cdfzonal_gpu_mean_device

     INTEGER(C_INT) FUNCTION cdfmhst_gpu_setup(nx, ny, nz, e1v, e3v, vmask1, atl, pac, ind) BIND(C, NAME='cdfmhst_gpu_setup')
       IMPORT :: C_INT, C_FLOAT, C_PTR
       INTEGER(C_INT), VALUE :: nx, ny, nz
       REAL(C_FLOAT), INTENT(in) :: e1v(*), e3v(*), vmask1(*)   ! e3v (npiglo,npjglo,npk) as read (cdfmhst.f90:331-334)
       TYPE(C_PTR), VALUE :: atl, pac, ind                  ! C_LOC of the basin masks, or all C_NULL_PTR
     END FUNCTION cdfmhst_gpu_setup

     INTEGER(C_INT) FUNCTION cdfmhst_gpu_record(zvt, zvs, zdim, heat, salt) BIND(C, NAME='cdfmhst_gpu_record')
       IMPORT :: C_INT, C_FLOAT, C_DOUBLE
       REAL(C_FLOAT), INTENT(in) :: zvt(*), zvs(*)          ! (npiglo,npjglo,npk)
       INTEGER(C_INT), VALUE :: zdim                        ! 1 with -Zdim
       REAL(C_DOUBLE), INTENT(out) :: heat(*), salt(*)      ! (npjglo,4,nlev): glo, atl, pac, ind raw zonal sums
     END FUNCTION cdfmhst_gpu_record

     ! -v/-t[-s] mode: V, T, S as read; the V-point products of cdfmhst.f90:313-323 are formed on the device
     INTEGER(C_INT) FUNCTION cdfmhst_gpu_record_vts(zv, zt, zs, zdim, heat, salt) BIND(C, NAME='cdfmhst_gpu_record_vts')
       IMPORT :: C_INT, C_FLOAT, C_DOUBLE
       REAL(C_FLOAT), INTENT(in) :: zv(*), zt(*), zs(*)     ! (npiglo,npjglo,npk)
       INTEGER(C_INT), VALUE :: zdim                        ! 1 with -Zdim
       REAL(C_DOUBLE), INTENT(out) :: heat(*), salt(*)      ! as cdfmhst_gpu_record
     END FUNCTION cdfmhst_gpu_record_vts

     ! record pipeline: submit on slot 0 .. cdfgpu_nslots()-1, fetch blocks; the records untouched until the fetch returns
     INTEGER(C_INT) FUNCTION cdfmhst_gpu_submit(slot, zvt, zvs, zdim) BIND(C, NAME='cdfmhst_gpu_submit')
       IMPORT :: C_INT, C_FLOAT
       INTEGER(C_INT), VALUE :: slot
       REAL(C_FLOAT), INTENT(in) :: zvt(*), zvs(*)          ! (npiglo,npjglo,npk), pinned
       INTEGER(C_INT), VALUE :: zdim                        ! 1 with -Zdim
     END FUNCTION cdfmhst_gpu_submit

     INTEGER(C_INT) FUNCTION cdfmhst_gpu_submit_vts(slot, zv, zt, zs, zdim) BIND(C, NAME='cdfmhst_gpu_submit_vts')
       IMPORT :: C_INT, C_FLOAT
       INTEGER(C_INT), VALUE :: slot
       REAL(C_FLOAT), INTENT(in) :: zv(*), zt(*), zs(*)     ! (npiglo,npjglo,npk), pinned
       INTEGER(C_INT), VALUE :: zdim                        ! 1 with -Zdim
     END FUNCTION cdfmhst_gpu_submit_vts

     INTEGER(C_INT) FUNCTION cdfmhst_gpu_fetch(slot, heat, salt) BIND(C, NAME='cdfmhst_gpu_fetch')
       IMPORT :: C_INT, C_DOUBLE
       INTEGER(C_INT), VALUE :: slot
       REAL(C_DOUBLE), INTENT(out) :: heat(*), salt(*)      ! as cdfmhst_gpu_record
     END FUNCTION cdfmhst_gpu_fetch

     INTEGER(C_INT) FUNCTION cdfmhst_gpu_teardown() BIND(C, NAME='cdfmhst_gpu_teardown')
       IMPORT :: C_INT
     END FUNCTION cdfmhst_gpu_teardown

     ! device-resident records, as cdfzonal_gpu_sum_device
     INTEGER(C_INT) FUNCTION cdfmhst_gpu_record_device(d_zvt, d_zvs, zdim, d_heat, d_salt, stream) &
          &                                           BIND(C, NAME='cdfmhst_gpu_record_device')
       IMPORT :: C_INT, C_PTR
       TYPE(C_PTR), VALUE :: d_zvt, d_zvs                   ! (npiglo,npjglo,npk) REAL(4)
       INTEGER(C_INT), VALUE :: zdim                        ! 1 with -Zdim
       TYPE(C_PTR), VALUE :: d_heat, d_salt                 ! (npjglo,4,nlev) REAL(8)
       TYPE(C_PTR), VALUE :: stream
     END FUNCTION cdfmhst_gpu_record_device

     INTEGER(C_INT) FUNCTION cdfmhst_gpu_record_vts_device(d_zv, d_zt, d_zs, zdim, d_heat, d_salt, stream) &
          &                                               BIND(C, NAME='cdfmhst_gpu_record_vts_device')
       IMPORT :: C_INT, C_PTR
       TYPE(C_PTR), VALUE :: d_zv, d_zt, d_zs               ! (npiglo,npjglo,npk) REAL(4)
       INTEGER(C_INT), VALUE :: zdim                        ! 1 with -Zdim
       TYPE(C_PTR), VALUE :: d_heat, d_salt                 ! (npjglo,4,nlev) REAL(8)
       TYPE(C_PTR), VALUE :: stream
     END FUNCTION cdfmhst_gpu_record_vts_device

     ! ---- cdftransig_xy3d (src/cdftransig_xy3d.f90:396-461): frame body on the GPU, accumulators resident -------------
     INTEGER(C_INT) FUNCTION cdftransig_gpu_setup(nx, ny, nz, nbins, pref, teos10, ds1min, ds1scalmin, nsigmax, itab, &
          &                                      e2u, e1v, e3u, e3v, lperio) BIND(C, NAME='cdftransig_gpu_setup')
       IMPORT :: C_INT, C_FLOAT, C_DOUBLE, C_PTR
       INTEGER(C_INT), VALUE :: nx, ny, nz, nbins, teos10, nsigmax, lperio
       REAL(C_FLOAT),  VALUE :: pref                        ! zpref
       REAL(C_DOUBLE), VALUE :: ds1min, ds1scalmin          ! ds1scalmin = MIN(ds1scalmin, ds1scal) (:213)
       INTEGER(C_INT), INTENT(in) :: itab(*)                ! (nsigmax), as built at :248-262
       REAL(C_FLOAT),  INTENT(in) :: e2u(*), e1v(*)         ! (npiglo,npjglo)
       TYPE(C_PTR), VALUE :: e3u, e3v                       ! C_LOC of (npiglo,npjglo,npk-1), or C_NULL_PTR with -vvl
     END FUNCTION cdftransig_gpu_setup

     INTEGER(C_INT) FUNCTION cdftransig_gpu_record(zu, zv, zt, zs, e3u_vvl, e3v_vvl, set_masks) &
          &                                       BIND(C, NAME='cdftransig_gpu_record')
       IMPORT :: C_INT, C_FLOAT, C_PTR
       REAL(C_FLOAT), INTENT(in) :: zu(*), zv(*), zt(*), zs(*)   ! one frame, (npiglo,npjglo,npk-1)
       TYPE(C_PTR), VALUE :: e3u_vvl, e3v_vvl               ! C_NULL_PTR unless -vvl
       INTEGER(C_INT), VALUE :: set_masks                   ! 1 for the frames of the first tag (jtag == 1, :410)
     END FUNCTION cdftransig_gpu_record

     ! frame pipeline on the first device, slots 0 .. nslots-1 of cdfgpu_init: frames accumulate in submission order
     INTEGER(C_INT) FUNCTION cdftransig_gpu_submit(slot, zu, zv, zt, zs, e3u_vvl, e3v_vvl, set_masks) &
          &                                       BIND(C, NAME='cdftransig_gpu_submit')
       IMPORT :: C_INT, C_FLOAT, C_PTR
       INTEGER(C_INT), VALUE :: slot
       REAL(C_FLOAT), INTENT(in) :: zu(*), zv(*), zt(*), zs(*)   ! one frame, pinned, untouched until cdftransig_gpu_wait(slot)
       TYPE(C_PTR), VALUE :: e3u_vvl, e3v_vvl               ! C_NULL_PTR unless -vvl
       INTEGER(C_INT), VALUE :: set_masks                   ! 1 for the frames of the first tag (jtag == 1, :410)
     END FUNCTION cdftransig_gpu_submit

     INTEGER(C_INT) FUNCTION cdftransig_gpu_wait(slot) BIND(C, NAME='cdftransig_gpu_wait')
       IMPORT :: C_INT
       INTEGER(C_INT), VALUE :: slot                        ! returns once the slot's frame is on the device
     END FUNCTION cdftransig_gpu_wait

     INTEGER(C_INT) FUNCTION cdftransig_gpu_fetch(dusigsig, dvsigsig) BIND(C, NAME='cdftransig_gpu_fetch')
       IMPORT :: C_INT, C_DOUBLE
       REAL(C_DOUBLE), INTENT(out) :: dusigsig(*), dvsigsig(*)   ! (npiglo,npjglo,nbins) raw sums
     END FUNCTION cdftransig_gpu_fetch

     INTEGER(C_INT) FUNCTION cdftransig_gpu_teardown() BIND(C, NAME='cdftransig_gpu_teardown')
       IMPORT :: C_INT
     END FUNCTION cdftransig_gpu_teardown

     ! a device-resident frame, as cdfzonal_gpu_sum_device; frames of every entry point accumulate in call order
     INTEGER(C_INT) FUNCTION cdftransig_gpu_record_device(d_zu, d_zv, d_zt, d_zs, d_e3u_vvl, d_e3v_vvl, set_masks, stream) &
          &                                              BIND(C, NAME='cdftransig_gpu_record_device')
       IMPORT :: C_INT, C_PTR
       TYPE(C_PTR), VALUE :: d_zu, d_zv, d_zt, d_zs         ! one frame, (npiglo,npjglo,npk-1) REAL(4)
       TYPE(C_PTR), VALUE :: d_e3u_vvl, d_e3v_vvl           ! C_NULL_PTR unless -vvl (read in place)
       INTEGER(C_INT), VALUE :: set_masks                   ! 1 for the frames of the first tag (jtag == 1, :410)
       TYPE(C_PTR), VALUE :: stream
     END FUNCTION cdftransig_gpu_record_device

     INTEGER(C_INT) FUNCTION cdftransig_gpu_fetch_device(d_dusigsig, d_dvsigsig, stream) &
          &                                             BIND(C, NAME='cdftransig_gpu_fetch_device')
       IMPORT :: C_INT, C_PTR
       TYPE(C_PTR), VALUE :: d_dusigsig, d_dvsigsig         ! (npiglo,npjglo,nbins) REAL(8), device-to-device copy of the raw sums
       TYPE(C_PTR), VALUE :: stream
     END FUNCTION cdftransig_gpu_fetch_device

     ! ---- cdfsigtrp: one section, replaces src/cdfsigtrp.f90:559-627 -------------------------------------------
     INTEGER(C_INT) FUNCTION cdfsigtrp_gpu_section(npts, npk, nk, eu, de3, ddepu, gdepw, ddepw_brk, zu, zt, zs, zmask, &
          &   kmode, refdep, kteos10, dsigma_min, dsigma_max, nbins, dsigma_lev, dsig, dhiso, dwtrp, dwtrpbin,      &
          &   dtrpbin) BIND(C, NAME='cdfsigtrp_gpu_section')
       IMPORT :: C_INT, C_FLOAT, C_DOUBLE, C_PTR
       INTEGER(C_INT), VALUE      :: npts, npk, nk, kmode, kteos10, nbins
       REAL(C_FLOAT),  VALUE      :: refdep
       REAL(C_DOUBLE), VALUE      :: dsigma_min, dsigma_max
       REAL(C_FLOAT),  INTENT(in) :: eu(*), de3(*)               ! (npts), (npts,npk) REAL(4) copy of de3
       REAL(C_DOUBLE), INTENT(in) :: ddepu(*)                    ! (npts,0:npk)
       REAL(C_FLOAT),  INTENT(in) :: gdepw(*)                    ! (npk)
       TYPE(C_PTR),    VALUE      :: ddepw_brk                   ! C_LOC of a REAL(4) (npts,npk) copy of ddepw (-brk), else C_NULL_PTR
       REAL(C_FLOAT),  INTENT(in) :: zu(*), zt(*), zs(*), zmask(*)
       REAL(C_DOUBLE), INTENT(out):: dsigma_lev(*)               ! (nbins+1)
       REAL(C_DOUBLE), INTENT(out):: dsig(*)                     ! (npts,0:nk): the first nk+1 rows of dsig(npts,0:npk)
       REAL(C_DOUBLE), INTENT(out):: dhiso(*), dwtrp(*)          ! (npts,nbins+1)
       REAL(C_DOUBLE), INTENT(out):: dwtrpbin(*), dtrpbin(*)     ! (npts,nbins), (nbins)
     END FUNCTION cdfsigtrp_gpu_section

     INTEGER(C_INT) FUNCTION cdfsigtrp_gpu_kernel_ms(ms) BIND(C, NAME='cdfsigtrp_gpu_kernel_ms')
       IMPORT :: C_INT, C_FLOAT
       REAL(C_FLOAT), INTENT(out) :: ms
     END FUNCTION cdfsigtrp_gpu_kernel_ms

     ! a list of sections cut from whole fields (the dens_section.dat boxes), cut and prepared on the device
     INTEGER(C_INT) FUNCTION cdfsigtrp_gpu_sections_setup(nx, ny, npk, nsec, ijbox, e1v, e2u, e3u, e3v, e3w, e3t_1d, e3w_1d, &
          &   gdept_1d, gdepw, zspu, zspv, zsps, kmode, refdep, kteos10, dsigma_min, dsigma_max, nbins, dsigma_lev,   &
          &   npts_out) BIND(C, NAME='cdfsigtrp_gpu_sections_setup')
       IMPORT :: C_INT, C_FLOAT, C_DOUBLE, C_PTR
       INTEGER(C_INT), VALUE      :: nx, ny, npk, nsec, kmode, kteos10, nbins
       INTEGER(C_INT), INTENT(in) :: ijbox(*)                   ! (4,nsec) imin imax jmin jmax
       TYPE(C_PTR),    VALUE      :: e1v, e2u                   ! C_LOC of (npiglo,npjglo) REAL(4), or C_NULL_PTR when unused
       TYPE(C_PTR),    VALUE      :: e3u, e3v, e3w              ! (npiglo,npjglo,npk) REAL(4), all three C_NULL_PTR with -full
       TYPE(C_PTR),    VALUE      :: e3t_1d, e3w_1d             ! (npk) REAL(4) for -full, else C_NULL_PTR
       REAL(C_FLOAT),  INTENT(in) :: gdept_1d(*), gdepw(*)      ! (npk)
       REAL(C_FLOAT),  VALUE      :: zspu, zspv, zsps, refdep
       REAL(C_DOUBLE), VALUE      :: dsigma_min, dsigma_max
       REAL(C_DOUBLE), INTENT(out):: dsigma_lev(*)              ! (nbins+1)
       INTEGER(C_INT), INTENT(out):: npts_out(*)                ! (nsec), 0 for a skipped section
     END FUNCTION cdfsigtrp_gpu_sections_setup

     ! one record of U, V, T, S in device memory (OpenACC host_data / CUDA Fortran), on `stream`
     INTEGER(C_INT) FUNCTION cdfsigtrp_gpu_sections_device(d_zu3d, d_zv3d, d_zt3d, d_zs3d, d_dtrpbin, d_nk, stream) &
          &                                               BIND(C, NAME='cdfsigtrp_gpu_sections_device')
       IMPORT :: C_INT, C_PTR
       TYPE(C_PTR), VALUE :: d_zu3d, d_zv3d, d_zt3d, d_zs3d   ! (npiglo,npjglo,npk) REAL(4); U / V C_NULL_PTR when no section needs it
       TYPE(C_PTR), VALUE :: d_dtrpbin                        ! (nbins,nsec) REAL(8), m3/s
       TYPE(C_PTR), VALUE :: d_nk                             ! (nsec) INTEGER(4) or C_NULL_PTR
       TYPE(C_PTR), VALUE :: stream
     END FUNCTION cdfsigtrp_gpu_sections_device

     INTEGER(C_INT) FUNCTION cdfsigtrp_gpu_teardown() BIND(C, NAME='cdfsigtrp_gpu_teardown')
       IMPORT :: C_INT
     END FUNCTION cdfsigtrp_gpu_teardown
  END INTERFACE

CONTAINS

  SUBROUTINE cdfgpu_check(kerr, cdwhere)
    !!---------------------------------------------------------------------
    !! Every non-zero status of the library is fatal for the tool: print the
    !! library's message and STOP 97 (the reference uses STOP 99 for usage /
    !! missing files and STOP 98 for NetCDF errors; 97 is new and GPU-specific).
    !!---------------------------------------------------------------------
    INTEGER(C_INT),   INTENT(in) :: kerr
    CHARACTER(LEN=*), INTENT(in) :: cdwhere
    CHARACTER(KIND=C_CHAR), POINTER :: cl_msg(:)
    INTEGER :: ji
    IF ( kerr == CDFGPU_OK ) RETURN
    CALL C_F_POINTER(cdfgpu_last_error(), cl_msg, (/512/))
    PRINT *, ' ERROR in ', TRIM(cdwhere), ' : libcdfgpu status ', kerr
    DO ji = 1, 512
       IF ( cl_msg(ji) == C_NULL_CHAR ) EXIT
       WRITE(*,'(a)', ADVANCE='NO') cl_msg(ji)
    END DO
    PRINT *
    STOP 97
  END SUBROUTINE cdfgpu_check

  FUNCTION cdfgpu_pinned_r4_3d(kpi, kpj, kpk) RESULT(ptab)
    !!---------------------------------------------------------------------
    !! Page-locked REAL(4) (kpi,kpj,kpk) buffer for NF90_GET_VAR to fill: the
    !! H2D copy of a record then runs asynchronously on the library's copy
    !! stream and overlaps the previous record's kernel.
    !!---------------------------------------------------------------------
    INTEGER(KIND=4), INTENT(in) :: kpi, kpj, kpk
    REAL(KIND=4), POINTER :: ptab(:,:,:)
    TYPE(C_PTR) :: cl_p
    cl_p = cdfgpu_pinned_alloc( INT(kpi,C_SIZE_T)*INT(kpj,C_SIZE_T)*INT(kpk,C_SIZE_T)*4_C_SIZE_T )
    IF ( .NOT. C_ASSOCIATED(cl_p) ) THEN
       PRINT *, ' ERROR : cdfgpu_pinned_alloc failed' ; STOP 97
    ENDIF
    CALL C_F_POINTER(cl_p, ptab, (/kpi, kpj, kpk/))
  END FUNCTION cdfgpu_pinned_r4_3d

  FUNCTION cdfgpu_pinned_i2_3d(kpi, kpj, kpk) RESULT(ktab)
    !!---------------------------------------------------------------------
    !! Page-locked INTEGER(2) (kpi,kpj,kpk) buffer for a packed record
    !! (getvar3d_i2_into): half the bytes of the REAL(4) record over PCIe,
    !! unpacked on the device (cdfgpu_set_input_packing).
    !!---------------------------------------------------------------------
    INTEGER(KIND=4), INTENT(in) :: kpi, kpj, kpk
    INTEGER(KIND=2), POINTER :: ktab(:,:,:)
    TYPE(C_PTR) :: cl_p
    cl_p = cdfgpu_pinned_alloc( INT(kpi,C_SIZE_T)*INT(kpj,C_SIZE_T)*INT(kpk,C_SIZE_T)*2_C_SIZE_T )
    IF ( .NOT. C_ASSOCIATED(cl_p) ) THEN
       PRINT *, ' ERROR : cdfgpu_pinned_alloc failed' ; STOP 97
    ENDIF
    CALL C_F_POINTER(cl_p, ktab, (/kpi, kpj, kpk/))
  END FUNCTION cdfgpu_pinned_i2_3d

END MODULE cdfgpu
