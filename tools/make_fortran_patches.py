#!/usr/bin/env python3
"""Generates cdftools_b200/fortran/patches/{cdfmoc,cdfmocsig,cdfsigtrp}.f90.patch: the call-site changes a CDFTOOLS maintainer applies
to the reference drivers so that the hot loop nests run on the GPU behind libcdfgpu's C ABI (INTEGRATION.md).

    python tools/make_fortran_patches.py /path/to/CDFTOOLS        # default $CDFTOOLS_REF

The patched drivers are assembled here from the reference sources by anchored edits and emitted as unified diffs: the
repository ships the DIFFS (what changes), never the reference's sources.  tools/apply_reference_patches.sh applies them to
a checkout and builds cdfmoc / cdfmocsig against libcdfgpu.so where a Fortran toolchain exists.
"""
import difflib
import os
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
if len(sys.argv) < 2 and not os.environ.get("CDFTOOLS_REF"):
    sys.exit("usage: make_fortran_patches.py /path/to/CDFTOOLS (or set CDFTOOLS_REF)")
REF = Path(sys.argv[1] if len(sys.argv) > 1 else os.environ["CDFTOOLS_REF"]) / "src"
OUT = ROOT / "cdftools_b200" / "fortran" / "patches"


def between(lines, start_pred, end_pred, start_from=0):
    """indices [i0, i1] of the first line matching start_pred (from start_from) and the first after it matching end_pred"""
    i0 = next(i for i in range(start_from, len(lines)) if start_pred(lines[i]))
    i1 = next(i for i in range(i0, len(lines)) if end_pred(lines[i]))
    return i0, i1


def insert_after(lines, pred, new, start_from=0):
    i = next(i for i in range(start_from, len(lines)) if pred(lines[i]))
    lines[i + 1:i + 1] = new
    return i + 1 + len(new)


def patch_cdfmoc(src):
    L = src.split("\n")
    insert_after(L, lambda l: l.strip() == "USE eos", [
        "  USE cdfgpu          ! ISO_C_BINDING interface of libcdfgpu.so (the B200 hot path)",
        "  USE cdfio_pinned    ! getvar3d_into : a whole record straight into a pinned buffer",
    ])
    insert_after(L, lambda l: l.startswith("  LOGICAL") and "ll_teos10" in l, [
        "",
        "  ! GPU hot path : record slots, read-ahead, pinned record buffers",
        "  TYPE t_pinned",
        "     REAL(KIND=4), DIMENSION(:,:,:), POINTER :: v => NULL(), t => NULL(), s => NULL()",
        "  END TYPE t_pinned",
        "  TYPE(t_pinned), DIMENSION(:), ALLOCATABLE   :: pin             ! one set of buffers per slot",
        "  INTEGER(KIND=4)                             :: nslot, nahead   ! record slots, records read ahead",
        "  INTEGER(KIND=4)                             :: jslot, jtr      ! slot / record index",
        "  INTEGER(KIND=2), DIMENSION(:,:,:), ALLOCATABLE :: iumask3d, itmask3d ! -decomp : masks of every level",
        "  LOGICAL                                     :: lnc4 = .FALSE.  ! -nc4 (DEV_TOOLS/tagnc4.tpl)",
    ])
    insert_after(L, lambda l: "CASE ( '-teos10')" in l, [
        "     CASE ('-nc4'   ) ; lnc4   = .TRUE.",
    ])
    # the time loop: everything from 'DO jt = 1, npt' up to the line before '     ! netcdf output' is replaced
    i0, i1 = between(L, lambda l: l.strip() == "DO jt = 1, npt", lambda l: l.strip() == "! netcdf output")
    gpu = '''  ! ---- GPU hot path (replaces the loop nests of the zonal integral, the vertical scan and the decomposition) ----
  CALL cdfgpu_check( cdfgpu_init(-1, 3), 'cdfgpu_init' )        ! $CDFGPU_DEVICES / $CDFGPU_SHARD : several GPUs
  DO jk = 1, npk
     e3v(:,:,jk) = get_e3v(jk,1)                                ! e3v masked with vmask, as before
  END DO
  CALL cdfgpu_check( cdfmoc_gpu_setup(npiglo, npjglo, npk, nbasins, e1v, e3v, ibmask), 'cdfmoc_gpu_setup' )
  IF ( ldec ) THEN
     ALLOCATE ( iumask3d(npiglo,npjglo,npk-1), itmask3d(npiglo,npjglo,npk-1) )
     DO jk = 1, npk-1
        iumask3d(:,:,jk) = getvar(cn_fmsk, cn_umask, jk, npiglo, npjglo)
        itmask3d(:,:,jk) = getvar(cn_fmsk, cn_tmask, jk, npiglo, npjglo)
     END DO
     ierr = 0 ; IF ( ll_teos10 ) ierr = 1
     CALL cdfgpu_check( cdfmoc_gpu_decomp_setup(ierr, e1u, gphiv, gdept, iumask3d, itmask3d), 'cdfmoc_gpu_decomp_setup' )
  ENDIF
  ! slots : every device has its own 3-deep pipeline; -vvl and -decomp keep one record in flight
  nslot = cdfgpu_nslots()
  IF ( lg_vvl .OR. ldec ) nslot = 1
  nahead = nslot - 1
  ALLOCATE ( pin(0:nslot-1) )
  DO jslot = 0, nslot-1
     pin(jslot)%v => cdfgpu_pinned_r4_3d(npiglo, npjglo, npk-1)
     IF ( ldec ) pin(jslot)%t => cdfgpu_pinned_r4_3d(npiglo, npjglo, npk-1)
     IF ( ldec ) pin(jslot)%s => cdfgpu_pinned_r4_3d(npiglo, npjglo, npk-1)
  END DO
  DO jtr = 1, MIN(nahead, npt)                                  ! records read ahead of the loop
     CALL read_and_submit(jtr)
  END DO

  DO jt = 1, npt
     IF ( lg_vvl .AND. jt > 1 ) THEN                            ! -vvl : the area field of this record
        DO jk = 1, npk
           e3v(:,:,jk) = get_e3v(jk,jt)
        END DO
        CALL cdfgpu_check( cdfmoc_gpu_set_e3v(e3v), 'cdfmoc_gpu_set_e3v' )
     ENDIF
     ! record jt+nahead goes to its device while record jt is being integrated
     IF ( jt + nahead <= npt ) CALL read_and_submit(jt + nahead)
     jslot = MOD(jt-1, nslot)
     IF ( ldec ) THEN
        CALL cdfgpu_check( cdfmoc_gpu_decomp_fetch(jslot, dmoc, dmoc_sh, dmoc_bt, dmoc_ag), 'cdfmoc_gpu_decomp_fetch' )
     ELSE
        CALL cdfgpu_check( cdfmoc_gpu_fetch(jslot, dmoc), 'cdfmoc_gpu_fetch' )
     ENDIF
'''.split("\n")
    L[i0:i1] = gpu
    # after the time loop: release
    i = next(i for i in range(len(L)) if L[i].strip() == "ierr = closeout(ncout)")
    L[i + 1:i + 1] = [
        "  CALL close_pinned_files()",
        "  CALL cdfgpu_check( cdfgpu_finalize(), 'cdfgpu_finalize' )",
    ]
    # internal procedure read_and_submit, in front of get_e3v
    i = next(i for i in range(len(L)) if L[i].strip().startswith("FUNCTION get_e3v"))
    L[i:i] = '''  SUBROUTINE read_and_submit (kt)
    !!---------------------------------------------------------------------
    !!                  ***  ROUTINE read_and_submit  ***
    !!
    !! ** Purpose :  read record kt into the pinned buffers of its slot and hand it to the GPU.
    !!               The H2D copy runs on a side stream and overlaps the kernel of the record before.
    !!----------------------------------------------------------------------
    INTEGER(KIND=4), INTENT(in) :: kt
    INTEGER(KIND=4)             :: islot
    !!----------------------------------------------------------------------
    islot = MOD(kt-1, nslot)
    CALL getvar3d_into(cf_vfil, cn_vomecrty, npiglo, npjglo, npk-1, pin(islot)%v, ktime=kt)
    IF ( ldec ) THEN
       CALL getvar3d_into(cf_tfil, cn_votemper, npiglo, npjglo, npk-1, pin(islot)%t, ktime=kt)
       CALL getvar3d_into(cf_sfil, cn_vosaline, npiglo, npjglo, npk-1, pin(islot)%s, ktime=kt)
       CALL cdfgpu_check( cdfmoc_gpu_decomp_submit(islot, kt, pin(islot)%v, pin(islot)%t, pin(islot)%s), 'cdfmoc_gpu_decomp_submit' )
    ELSE
       CALL cdfgpu_check( cdfmoc_gpu_submit(islot, kt, pin(islot)%v), 'cdfmoc_gpu_submit' )
    ENDIF
  END SUBROUTINE read_and_submit

'''.split("\n")
    # -nc4 in CreateOutput
    for i, l in enumerate(L):
        if "ncout = create      ( cf_moc,  'none',    1, npjglo, npk, cdep=cn_vdepthw )" in l:
            L[i] = "    ncout = create      ( cf_moc,  'none',    1, npjglo, npk, cdep=cn_vdepthw, ld_nc4=lnc4 )"
        if "ierr  = createvar   ( ncout,   stypvar,   nvarout,   ipk, id_varout, cdglobal=TRIM(cglobal)" in l:
            L[i] = "    ierr  = createvar   ( ncout,   stypvar,   nvarout,   ipk, id_varout, cdglobal=TRIM(cglobal), ld_nc4=lnc4 )"
    return "\n".join(L)


def patch_cdfmocsig(src):
    L = src.split("\n")
    insert_after(L, lambda l: l.strip() == "USE modutils", [
        "  USE cdfgpu          ! ISO_C_BINDING interface of libcdfgpu.so (the B200 hot path)",
        "  USE cdfio_pinned    ! getvar3d_into : a whole record straight into a pinned buffer",
    ])
    insert_after(L, lambda l: l.startswith("  LOGICAL") and "ll_teos10" in l, [
        "",
        "  ! GPU hot path : record slots, read-ahead, pinned record buffers",
        "  TYPE t_pinned",
        "     REAL(KIND=4), DIMENSION(:,:,:), POINTER :: v => NULL(), t => NULL(), s => NULL(), eiv => NULL(), e3 => NULL()",
        "  END TYPE t_pinned",
        "  TYPE(t_pinned), DIMENSION(:), ALLOCATABLE       :: pin                  ! one set of buffers per slot",
        "  REAL(KIND=4), DIMENSION(:,:,:), ALLOCATABLE, TARGET :: e3v3d            ! e3v of every level (NOT masked)",
        "  TYPE(C_PTR)                                     :: cl_eiv, cl_e3        ! optional fields of a record (or C_NULL_PTR)",
        "  REAL(KIND=4), DIMENSION(:),     ALLOCATABLE     :: gdept1d              ! deptht for -isodep",
        "  INTEGER(KIND=4)                                 :: nslot, nahead        ! record slots, records read ahead",
        "  INTEGER(KIND=4)                                 :: jslot, jtr, ieos     ! slot / record index, EOS selector",
        "  LOGICAL                                         :: lnc4 = .FALSE.       ! -nc4 (DEV_TOOLS/tagnc4.tpl)",
    ])
    insert_after(L, lambda l: "CASE ('-verbose')" in l, [
        "     CASE ('-nc4'    ) ; lnc4    = .TRUE.",
    ])
    i0, i1 = between(L, lambda l: l.strip() == "DO jt=1, npt", lambda l: l.strip().startswith("! netcdf output"))
    gpu = '''  ! ---- GPU hot path (replaces the loop nest : scrub, area, EOS, binning, scatter-add, bin cumsum) ----
  CALL cdfgpu_check( cdfgpu_init(-1, 3), 'cdfgpu_init' )        ! $CDFGPU_DEVICES / $CDFGPU_SHARD : several GPUs
  ieos = CDFGPU_EOS_EOS80
  IF ( ll_teos10 ) ieos = CDFGPU_EOS_TEOS10
  IF ( lntr      ) ieos = CDFGPU_EOS_NEUTRAL
  ALLOCATE ( e3v3d(npiglo,npjglo,npk) )
  IF ( .NOT. lg_vvl ) THEN                                      ! e3v of every level, NOT masked, as the loop read it
     DO jk = 1, npk-1
        IF ( lfull ) THEN ; e3v3d(:,:,jk) = e31d(jk)
        ELSE              ; e3v3d(:,:,jk) = getvar(cn_fe3v, cn_ve3v, jk, npiglo, npjglo, ktime=1, ldiom=.TRUE.)
        ENDIF
     END DO
     e3v3d(:,:,npk) = 0.
     CALL cdfgpu_check( cdfmocsig_gpu_setup(npiglo, npjglo, npk, nbasins, nbins, sigmin, sigstp, pref, ieos, e1v,         &
          &             C_LOC(e3v3d), ibmask, zspv, zspt, zsps, 0, npjglo), 'cdfmocsig_gpu_setup' )
  ELSE                                                          ! -vvl : every record brings its own e3v
     CALL cdfgpu_check( cdfmocsig_gpu_setup(npiglo, npjglo, npk, nbasins, nbins, sigmin, sigstp, pref, ieos, e1v,         &
          &             C_NULL_PTR,   ibmask, zspv, zspt, zsps, 0, npjglo), 'cdfmocsig_gpu_setup' )
  ENDIF
  IF ( lisodep ) THEN
     ALLOCATE ( gdept1d(npk) )
     gdept1d(:) = getvare3(cn_fzgr, cn_gdept, npk)              ! the library forms gdep = -gdept itself
     CALL cdfgpu_check( cdfmocsig_gpu_set_isodep(gdept1d), 'cdfmocsig_gpu_set_isodep' )
  ENDIF
  nslot = cdfgpu_nslots()
  IF ( lg_vvl ) nslot = 1                                       ! the area field is rebuilt per record
  nahead = nslot - 1
  ALLOCATE ( pin(0:nslot-1) )
  DO jslot = 0, nslot-1
     pin(jslot)%v => cdfgpu_pinned_r4_3d(npiglo, npjglo, npk-1)
     pin(jslot)%t => cdfgpu_pinned_r4_3d(npiglo, npjglo, npk-1)
     pin(jslot)%s => cdfgpu_pinned_r4_3d(npiglo, npjglo, npk-1)
     IF ( leiv   ) pin(jslot)%eiv => cdfgpu_pinned_r4_3d(npiglo, npjglo, npk-1)
     IF ( lg_vvl ) pin(jslot)%e3  => cdfgpu_pinned_r4_3d(npiglo, npjglo, npk-1)
  END DO
  DO jtr = 1, MIN(nahead, npt)                                  ! records read ahead of the loop
     CALL read_and_submit(jtr)
  END DO

  DO jt=1, npt
     IF (lprint) PRINT *,' working at record ',jt
     ! record jt+nahead goes to its device while record jt is being binned
     IF ( jt + nahead <= npt ) CALL read_and_submit(jt + nahead)
     jslot = MOD(jt-1, nslot)
     CALL cdfgpu_check( cdfmocsig_gpu_fetch(jslot, dmoc), 'cdfmocsig_gpu_fetch' )
     IF ( lisodep ) CALL cdfgpu_check( cdfmocsig_gpu_fetch_isodep(jslot, depi), 'cdfmocsig_gpu_fetch_isodep' )

'''.split("\n")
    L[i0:i1] = gpu
    i = next(i for i in range(len(L)) if L[i].strip() == "ierr = closeout(ncout)")
    L[i + 1:i + 1] = [
        "  CALL close_pinned_files()",
        "  CALL cdfgpu_check( cdfgpu_finalize(), 'cdfgpu_finalize' )",
    ]
    i = next(i for i in range(len(L)) if L[i].strip().startswith("SUBROUTINE CreateOutputFile"))
    L[i:i] = '''  SUBROUTINE read_and_submit (kt)
    !!---------------------------------------------------------------------
    !!                  ***  ROUTINE read_and_submit  ***
    !!
    !! ** Purpose :  read record kt (raw file values : the missing-value scrub runs on the GPU) into the
    !!               pinned buffers of its slot and hand it to the GPU.
    !!----------------------------------------------------------------------
    INTEGER(KIND=4), INTENT(in) :: kt
    INTEGER(KIND=4)             :: islot
    !!----------------------------------------------------------------------
    islot = MOD(kt-1, nslot)
    CALL getvar3d_into(cf_vfil, cn_vomecrty, npiglo, npjglo, npk-1, pin(islot)%v, ktime=kt)
    CALL getvar3d_into(cf_tfil, cn_votemper, npiglo, npjglo, npk-1, pin(islot)%t, ktime=kt)
    CALL getvar3d_into(cf_sfil, cn_vosaline, npiglo, npjglo, npk-1, pin(islot)%s, ktime=kt)
    IF ( leiv   ) CALL getvar3d_into(cf_vfil, cn_vomeeivv, npiglo, npjglo, npk-1, pin(islot)%eiv, ktime=kt)
    IF ( lg_vvl ) CALL getvar3d_into(cn_fe3v, cn_ve3vvvl,  npiglo, npjglo, npk-1, pin(islot)%e3,  ktime=kt)
    cl_eiv = C_NULL_PTR ; IF ( leiv   ) cl_eiv = C_LOC( pin(islot)%eiv )
    cl_e3  = C_NULL_PTR ; IF ( lg_vvl ) cl_e3  = C_LOC( pin(islot)%e3  )
    CALL cdfgpu_check( cdfmocsig_gpu_submit(islot, kt, pin(islot)%v, pin(islot)%t, pin(islot)%s, cl_eiv, cl_e3), &
         &             'cdfmocsig_gpu_submit' )
  END SUBROUTINE read_and_submit

'''.split("\n")
    for i, l in enumerate(L):
        if "ncout = create      (cf_moc, 'none', 1,      npjglo, nbins,  cdep='sigma')" in l:
            L[i] = "    ncout = create      (cf_moc, 'none', 1,      npjglo, nbins,  cdep='sigma', ld_nc4=lnc4)"
        if "ierr  = createvar   (ncout,  stypvar, nvaro, ipk ,id_varout, cdglobal=cglobal)" in l:
            L[i] = "    ierr  = createvar   (ncout,  stypvar, nvaro, ipk ,id_varout, cdglobal=cglobal, ld_nc4=lnc4)"
    return "\n".join(L)


def patch_cdfsigtrp(src):
    L = src.split("\n")
    insert_after(L, lambda l: l.strip().startswith("USE eos"), [
        "  USE cdfgpu          ! ISO_C_BINDING interface of libcdfgpu.so (the B200 hot path)",
    ])
    insert_after(L, lambda l: l.startswith("  LOGICAL") and "ll_teos10" in l, [
        "",
        "  ! GPU hot path : REAL(4) copies the library takes, per-section result",
        "  INTEGER(KIND=4)                             :: imode, iteos10        ! density mode, TEOS10 flag",
        "  REAL(KIND=4), DIMENSION(:,:), ALLOCATABLE         :: zde3            ! de3 holds REAL(4) file values",
        "  REAL(KIND=4), DIMENSION(:,:), ALLOCATABLE, TARGET :: zdepw           ! -brk : w depths of every column",
        "  REAL(KIND=8), DIMENSION(:),   ALLOCATABLE         :: dtrpbin_sec     ! binned transport of the section",
        "  TYPE(C_PTR)                                       :: pdepw",
    ])
    insert_after(L, lambda l: l.strip() == "!! *  Main loop on sections", [
        "  CALL cdfgpu_check( cdfgpu_init(-1, 1), 'cdfgpu_init' )",
        "  ALLOCATE ( dtrpbin_sec(nbins) )",
    ])
    i0, i1 = between(L, lambda l: l.strip() == "! compute density only for wet points",
                     lambda l: l.strip() == "! output of the code for 1 section")
    gpu = '''     ! ---- GPU hot path (replaces the density, isopycnal depth, cumulated and binned transport loop nests) ----
     ALLOCATE ( zde3(npts,npk), zdepw(npts,npk) )
     zde3(:,:) = REAL(de3(:,:))
     pdepw     = C_NULL_PTR
     IF ( lbrk ) THEN                        ! in broken line gdepw is not available as 1d array
        zdepw(:,:) = REAL(ddepw(:,1:npk))
        pdepw      = C_LOC(zdepw)
     ENDIF
     imode = 0                               ! sigmai(refdep) ; sigma0 when refdep = 0
     IF ( lntr           ) imode = 1         ! neutral density
     IF ( refdep == -10. ) imode = 2         ! -temp
     iteos10 = 0 ; IF ( ll_teos10 ) iteos10 = 1
     CALL cdfgpu_check( cdfsigtrp_gpu_section(npts, npk, nk, eu, zde3, ddepu, gdepw, pdepw, zu, zt, zs, zmask,   &
          &   imode, refdep, iteos10, dsigma_min, dsigma_max, nbins, dsigma_lev, dsig, dhiso, dwtrp, dwtrpbin,   &
          &   dtrpbin_sec), 'cdfsigtrp_gpu_section' )
     dtrpbin(jsec,:) = dtrpbin_sec(:)
     DEALLOCATE ( zde3, zdepw )
'''.split("\n")
    L[i0:i1] = gpu
    insert_after(L, lambda l: l.strip() == "END DO   ! next section", [
        "  CALL cdfgpu_check( cdfgpu_finalize(), 'cdfgpu_finalize' )",
    ])
    return "\n".join(L)


def main():
    OUT.mkdir(parents=True, exist_ok=True)
    for name, fn in (("cdfmoc.f90", patch_cdfmoc), ("cdfmocsig.f90", patch_cdfmocsig), ("cdfsigtrp.f90", patch_cdfsigtrp)):
        a = (REF / name).read_text()
        b = fn(a)
        d = difflib.unified_diff(a.split("\n"), b.split("\n"), "a/src/" + name, "b/src/" + name, lineterm="", n=3)
        txt = "\n".join(d) + "\n"
        (OUT / (name + ".patch")).write_text(txt)
        print(name, ":", sum(1 for l in txt.split("\n") if l.startswith("+") and not l.startswith("+++")), "lines added,",
              sum(1 for l in txt.split("\n") if l.startswith("-") and not l.startswith("---")), "removed")


if __name__ == "__main__":
    main()
