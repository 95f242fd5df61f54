MODULE cdfio_pinned
  !!======================================================================
  !!                     ***  MODULE  cdfio_pinned  ***
  !! Record readers for the GPU hot path: a whole (x,y,z) record of one time
  !! frame goes STRAIGHT into a caller-supplied array -- in practice the
  !! page-locked buffer obtained from cdfgpu_pinned_alloc and mapped with
  !! c_f_pointer (cdfgpu_pinned_r4_3d in module cdfgpu) -- with ONE
  !! NF90_GET_VAR, and the file stays open from record to record.
  !!
  !! Why a new routine: every reader of cdfio returns its array as a FUNCTION
  !! RESULT (getvar, src/cdfio.F90:1425-1609; getvar3d, :1611-1715), i.e. in a
  !! compiler temporary that is then copied into the destination, and both
  !! re-open and close the file on every call (getvar: once per LEVEL).  The
  !! record pipeline of libcdfgpu needs the data in pinned memory without that
  !! extra copy, and cdfmoc / cdfmocsig read npk-1 levels per record.
  !!
  !! getvar3d_into is the subroutine twin of getvar3d: same arguments, same
  !! post-processing (scale_factor, add_offset, savelog10, applied where the
  !! value is not the missing value, in the reference's order), same error
  !! behaviour (message + STOP 98).
  !!
  !! NOTE: not compiled in the build image of this repository (no Fortran
  !! compiler, no netcdf-fortran there); standard Fortran 2003 + netcdf-fortran.
  !!======================================================================
  USE netcdf
  USE cdfio, ONLY : getspval
  IMPLICIT NONE
  PRIVATE

  INTEGER(KIND=4), PARAMETER :: jp_maxopen = 16            ! files kept open at a time
  INTEGER(KIND=4)            :: nopen = 0                  ! number of cached files
  CHARACTER(LEN=256), DIMENSION(jp_maxopen) :: cfcache = ' ' ! their names
  INTEGER(KIND=4),    DIMENSION(jp_maxopen) :: ncache = -1   ! their netcdf ids

  PUBLIC :: getvar3d_into      ! one (kpi,kpj,kpz) block of one time frame into ptab
  PUBLIC :: getvar3d_i2_into   ! the same for a packed INTEGER(2) variable, left packed
  PUBLIC :: close_pinned_files ! close the files getvar3d_into keeps open

CONTAINS

  INTEGER(KIND=4) FUNCTION ncid_of ( cdfile )
    !!---------------------------------------------------------------------
    !!                  ***  FUNCTION ncid_of  ***
    !!
    !! ** Purpose :  netcdf id of cdfile, opening it on first use
    !!----------------------------------------------------------------------
    CHARACTER(LEN=*), INTENT(in) :: cdfile
    INTEGER(KIND=4) :: jf, istatus
    !!----------------------------------------------------------------------
    DO jf = 1, nopen
       IF ( TRIM(cfcache(jf)) == TRIM(cdfile) ) THEN
          ncid_of = ncache(jf)
          RETURN
       ENDIF
    END DO
    IF ( nopen == jp_maxopen ) THEN    ! recycle the oldest entry
       istatus = NF90_CLOSE( ncache(1) )
       cfcache(1:jp_maxopen-1) = cfcache(2:jp_maxopen)
       ncache (1:jp_maxopen-1) = ncache (2:jp_maxopen)
       nopen = nopen - 1
    ENDIF
    nopen = nopen + 1
    istatus = NF90_OPEN( cdfile, NF90_NOWRITE, ncache(nopen) )
    IF ( istatus /= NF90_NOERR ) THEN
       PRINT *, ' ERROR in getvar3d_into : cannot open ', TRIM(cdfile)
       PRINT *, TRIM( NF90_STRERROR(istatus) )
       STOP 98
    ENDIF
    cfcache(nopen) = cdfile
    ncid_of = ncache(nopen)
  END FUNCTION ncid_of

  SUBROUTINE getvar3d_into ( cdfile, cdvar, kpi, kpj, kpz, ptab, kimin, kjmin, kkmin, ktime )
    !!---------------------------------------------------------------------
    !!                  ***  ROUTINE getvar3d_into  ***
    !!
    !! ** Purpose :  Read the 3D REAL block cdvar(kimin:, kjmin:, kkmin:, ktime)
    !!               of size (kpi,kpj,kpz) from cdfile into ptab.
    !!
    !! ** Method  :  As getvar3d (src/cdfio.F90:1611-1715), but the data go
    !!               to the array the caller supplies, and the file is not
    !!               re-opened for every call.
    !!----------------------------------------------------------------------
    CHARACTER(LEN=*),                     INTENT(in)  :: cdfile
    CHARACTER(LEN=*),                     INTENT(in)  :: cdvar
    INTEGER(KIND=4),                      INTENT(in)  :: kpi, kpj, kpz
    REAL(KIND=4), DIMENSION(kpi,kpj,kpz), INTENT(out) :: ptab          ! explicit shape: contiguous, no temporary
    INTEGER(KIND=4), OPTIONAL,            INTENT(in)  :: kimin, kjmin, kkmin
    INTEGER(KIND=4), OPTIONAL,            INTENT(in)  :: ktime         ! if missing 1 is assumed

    INTEGER(KIND=4), DIMENSION(4) :: istart, icount
    INTEGER(KIND=4)               :: incid, id_var, istatus
    INTEGER(KIND=4)               :: iimin, ijmin, ikmin, itime, ilog
    REAL(KIND=4)                  :: sf, ao             ! scale factor and add_offset
    REAL(KIND=4)                  :: spval              ! missing value
    LOGICAL                       :: llog, lsf, lao
    !!----------------------------------------------------------------------
    iimin = 1 ; ijmin = 1 ; ikmin = 1 ; itime = 1
    IF ( PRESENT(kimin) ) iimin = kimin
    IF ( PRESENT(kjmin) ) ijmin = kjmin
    IF ( PRESENT(kkmin) ) ikmin = kkmin
    IF ( PRESENT(ktime) ) itime = ktime
    llog = .FALSE. ; lsf = .FALSE. ; lao = .FALSE.
    sf = 1. ; ao = 0.

    incid   = ncid_of( cdfile )
    istatus = NF90_INQ_VARID( incid, cdvar, id_var )
    IF ( istatus /= NF90_NOERR ) THEN
       PRINT *, ' ERROR in getvar3d_into : no variable ', TRIM(cdvar), ' in ', TRIM(cdfile)
       STOP 98
    ENDIF
    istart = (/ iimin, ijmin, ikmin, itime /)
    icount = (/ kpi,   kpj,   kpz,   1     /)

    spval = getspval( cdfile, cdvar )     ! tries the usual spellings of the missing-value attribute

    istatus = NF90_INQUIRE_ATTRIBUTE( incid, id_var, 'savelog10' )
    IF ( istatus == NF90_NOERR ) THEN
       istatus = NF90_GET_ATT( incid, id_var, 'savelog10', ilog )
       IF ( ilog /= 0 ) llog = .TRUE.
    ENDIF
    istatus = NF90_INQUIRE_ATTRIBUTE( incid, id_var, 'scale_factor' )
    IF ( istatus == NF90_NOERR ) THEN
       istatus = NF90_GET_ATT( incid, id_var, 'scale_factor', sf )
       IF ( sf /= 1. ) lsf = .TRUE.
    ENDIF
    istatus = NF90_INQUIRE_ATTRIBUTE( incid, id_var, 'add_offset' )
    IF ( istatus == NF90_NOERR ) THEN
       istatus = NF90_GET_ATT( incid, id_var, 'add_offset', ao )
       IF ( ao /= 0. ) lao = .TRUE.
    ENDIF

    istatus = NF90_GET_VAR( incid, id_var, ptab, start=istart, count=icount )
    IF ( istatus /= NF90_NOERR ) THEN
       PRINT *, ' Problem in getvar3d_into for ', TRIM(cdvar)
       PRINT *, TRIM( NF90_STRERROR(istatus) )
       STOP 98
    ENDIF

    ! Caution : order does matter (as in getvar3d)
    IF ( lsf  )  WHERE ( ptab /= spval )  ptab = ptab * sf
    IF ( lao  )  WHERE ( ptab /= spval )  ptab = ptab + ao
    IF ( llog )  WHERE ( ptab /= spval )  ptab = 10**ptab

  END SUBROUTINE getvar3d_into

  SUBROUTINE getvar3d_i2_into ( cdfile, cdvar, kpi, kpj, kpz, ktab, psf, pao, pspval, ldlog, kimin, kjmin, kkmin, ktime )
    !!---------------------------------------------------------------------
    !!                  ***  ROUTINE getvar3d_i2_into  ***
    !!
    !! ** Purpose :  Read the 3D block cdvar(kimin:, kjmin:, kkmin:, ktime) of
    !!               a packed (NC_SHORT, cdf16bit) variable into the INTEGER(2)
    !!               array ktab, WITHOUT unpacking it: the GPU does that
    !!               (cdfgpu_set_input_packing with psf, pao, pspval).
    !!
    !! ** Method  :  One NF90_GET_VAR into ktab; no post-processing.  psf, pao,
    !!               pspval are what getvar3d_into would apply (1., 0. when the
    !!               attribute is absent); ldlog is .TRUE. when savelog10 is set,
    !!               in which case the caller must read the variable with
    !!               getvar3d_into instead (10** stays on the host).
    !!----------------------------------------------------------------------
    CHARACTER(LEN=*),                        INTENT(in)  :: cdfile
    CHARACTER(LEN=*),                        INTENT(in)  :: cdvar
    INTEGER(KIND=4),                         INTENT(in)  :: kpi, kpj, kpz
    INTEGER(KIND=2), DIMENSION(kpi,kpj,kpz), INTENT(out) :: ktab       ! explicit shape: contiguous, no temporary
    REAL(KIND=4),                            INTENT(out) :: psf, pao, pspval
    LOGICAL,                                 INTENT(out) :: ldlog
    INTEGER(KIND=4), OPTIONAL,               INTENT(in)  :: kimin, kjmin, kkmin
    INTEGER(KIND=4), OPTIONAL,               INTENT(in)  :: ktime      ! if missing 1 is assumed

    INTEGER(KIND=4), DIMENSION(4) :: istart, icount
    INTEGER(KIND=4)               :: incid, id_var, istatus
    INTEGER(KIND=4)               :: iimin, ijmin, ikmin, itime, ilog
    !!----------------------------------------------------------------------
    iimin = 1 ; ijmin = 1 ; ikmin = 1 ; itime = 1
    IF ( PRESENT(kimin) ) iimin = kimin
    IF ( PRESENT(kjmin) ) ijmin = kjmin
    IF ( PRESENT(kkmin) ) ikmin = kkmin
    IF ( PRESENT(ktime) ) itime = ktime
    ldlog = .FALSE.
    psf = 1. ; pao = 0.

    incid   = ncid_of( cdfile )
    istatus = NF90_INQ_VARID( incid, cdvar, id_var )
    IF ( istatus /= NF90_NOERR ) THEN
       PRINT *, ' ERROR in getvar3d_i2_into : no variable ', TRIM(cdvar), ' in ', TRIM(cdfile)
       STOP 98
    ENDIF
    istart = (/ iimin, ijmin, ikmin, itime /)
    icount = (/ kpi,   kpj,   kpz,   1     /)

    pspval = getspval( cdfile, cdvar )

    istatus = NF90_INQUIRE_ATTRIBUTE( incid, id_var, 'savelog10' )
    IF ( istatus == NF90_NOERR ) THEN
       istatus = NF90_GET_ATT( incid, id_var, 'savelog10', ilog )
       IF ( ilog /= 0 ) ldlog = .TRUE.
    ENDIF
    istatus = NF90_INQUIRE_ATTRIBUTE( incid, id_var, 'scale_factor' )
    IF ( istatus == NF90_NOERR ) istatus = NF90_GET_ATT( incid, id_var, 'scale_factor', psf )
    istatus = NF90_INQUIRE_ATTRIBUTE( incid, id_var, 'add_offset' )
    IF ( istatus == NF90_NOERR ) istatus = NF90_GET_ATT( incid, id_var, 'add_offset', pao )

    istatus = NF90_GET_VAR( incid, id_var, ktab, start=istart, count=icount )
    IF ( istatus /= NF90_NOERR ) THEN
       PRINT *, ' Problem in getvar3d_i2_into for ', TRIM(cdvar)
       PRINT *, TRIM( NF90_STRERROR(istatus) )
       STOP 98
    ENDIF

  END SUBROUTINE getvar3d_i2_into

  SUBROUTINE close_pinned_files ()
    !!---------------------------------------------------------------------
    !!                  ***  ROUTINE close_pinned_files  ***
    !!
    !! ** Purpose :  close every file getvar3d_into has opened
    !!----------------------------------------------------------------------
    INTEGER(KIND=4) :: jf, istatus
    !!----------------------------------------------------------------------
    DO jf = 1, nopen
       istatus = NF90_CLOSE( ncache(jf) )
    END DO
    nopen = 0
    cfcache(:) = ' '
    ncache(:)  = -1
  END SUBROUTINE close_pinned_files

END MODULE cdfio_pinned
