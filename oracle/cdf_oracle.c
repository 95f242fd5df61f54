/*
 * cdf_oracle.c -- CPU restatement of the cdfmoc / cdfmocsig hot path of meom-group/CDFTOOLS.
 *
 * THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may load it.  The product path
 * (cdftools_b200/csrc + libcdfgpu.so) never calls anything in this file and has no CPU fallback.
 *
 * Pinning status: the reference carries no golden vectors or tests for the zonal integral,
 * the scan, the binning or the scatter (SURVEY.md section 4) and no Fortran compiler or
 * NetCDF library exists in this image, so the reference itself cannot be run here:
 *   - EOS routines (sigmai_dep, sigmantr): PINNED by the three check values printed in the
 *     reference's comments (src/eos.f90:646,817,820) -- see tests/test_oracle_eos.py.
 *   - zonal integral / scan / binning / scatter: PARITY UNPINNED by the reference; pinned only by
 *     (i) an independent NumPy restatement agreeing bit for bit (oracle/np_oracle.py),
 *     (ii) a hand-computed 4x3x3 case, (iii) algebraic property tests.
 *
 * Arithmetic rules (SURVEY.md App. A): REAL(4) temporaries are `float`, REAL(8) are `double`,
 * products associate left to right exactly as written in the Fortran, sums run sequentially in the
 * reference loop order, no FMA contraction (compile with -ffp-contract=off, no -ffast-math).
 *
 * Memory layout: Fortran column-major arrays are passed flat, first index fastest:
 *   e1v(nx,ny)        -> e1v[j*nx+i]
 *   e3v(nx,ny,nz)     -> e3v[(k*ny+j)*nx+i]
 *   ibmask(nb,nx,ny)  -> ibmask[(j*nx+i)*nb+b]          (INTEGER(2), basin fastest)
 *   dmoc(nb,ny,nz)    -> dmoc[(k*ny+j)*nb+b]            (cdfmoc.f90:287)
 *   dmoc(nb,nbins,ny) -> dmoc[(j*nbins+bin)*nb+b]       (cdfmocsig.f90:313)
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "../include/cdf_eos_coeffs.h"

#define CDF_EOS_EOS80 0
#define CDF_EOS_TEOS10 1
#define CDF_EOS_NEUTRAL 2

int oracle_abi_version(void) { return 1; }

void oracle_set_num_threads(int n)
{
    if (n > 0) omp_set_num_threads(n);
}

int oracle_num_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

/* ---------------------------------------------------------------------------------------------
 * a1. basin mask assembly -- src/cdfmoc.f90:325-336 (cdfmocsig.f90:347-359).
 * getvar() returns REAL(4); assignment to INTEGER(2) truncates toward zero.
 * Order: 1 global(vmask k=1), 2 atl, 3 indo-pacific = min(1, pac+ind), 4 ind, 5 pac.
 * The i=1 and i=nx columns of the GLOBAL mask are zeroed (periodic overlap).
 * In cdfmocsig the zeroing sits inside IF(lbas) (:356-358): `zero_edges_always`=0 reproduces that.
 * ------------------------------------------------------------------------------------------- */
void oracle_basin_masks(int nx, int ny, int nb, const float *vmask1, const float *atl, const float *ind,
                        const float *pac, int zero_edges, int16_t *ibmask)
{
    for (int j = 0; j < ny; ++j)
        for (int i = 0; i < nx; ++i) {
            size_t c = (size_t)j * nx + i;
            int16_t *m = ibmask + c * nb;
            m[0] = (int16_t)vmask1[c];
            if (nb >= 5) {
                m[1] = (int16_t)atl[c];
                m[3] = (int16_t)ind[c];
                m[4] = (int16_t)pac[c];
                m[2] = (int16_t)(m[4] + m[3]);
                if (m[2] > 0) m[2] = 1;
            }
        }
    if (zero_edges)
        for (int j = 0; j < ny; ++j) {
            ibmask[((size_t)j * nx + 0) * nb] = 0;
            ibmask[((size_t)j * nx + (nx - 1)) * nb] = 0;
        }
}

/* ---------------------------------------------------------------------------------------------
 * a2. get_e3v -- src/cdfmoc.f90:590-594: e3v(:,:) = e3v_file(:,:) * ivmask(:,:)
 * ivmask is INTEGER(2) (truncated from the REAL(4) getvar result); product is REAL(4).
 * ------------------------------------------------------------------------------------------- */
void oracle_mask_e3v(size_t n, const float *e3v_file, const float *vmask, float *e3m)
{
    for (size_t c = 0; c < n; ++c) {
        int16_t iv = (int16_t)vmask[c];
        e3m[c] = e3v_file[c] * (float)iv;
    }
}

/* ---------------------------------------------------------------------------------------------
 * a3 + a4. cdfmoc record -- src/cdfmoc.f90:352-388.
 *   dmoc(b,j,k) = dmoc(b,j,k) - e1v(i,j)*e3v(i,j,k)*ibmask(b,i,j)*zv(i,j)*1.d0     (:373-374)
 * The REAL(4)*REAL(4)*INTEGER(2)*REAL(4) chain is evaluated left to right in REAL(4); *1.d0 widens.
 * zv holds levels 1..nz-1 only (level nz is never read, :355).  No missing-value scrub (:357).
 *   dmoc(:,j,k) = dmoc(:,j,k+1) + dmoc(:,j,k)/1.d6, k = nz-1..1                      (:385)
 * ------------------------------------------------------------------------------------------- */
void oracle_cdfmoc_record(int nx, int ny, int nz, int nb, const float *e1v, const float *e3m,
                          const int16_t *ibmask, const float *zv, double *dmoc)
{
    memset(dmoc, 0, sizeof(double) * (size_t)nb * ny * nz);
    for (int k = 0; k < nz - 1; ++k)
        for (int b = 0; b < nb; ++b) {
#pragma omp parallel for schedule(runtime)
            for (int j = 0; j < ny; ++j) {
                double acc = dmoc[((size_t)k * ny + j) * nb + b];
                const float *pe1 = e1v + (size_t)j * nx;
                const float *pe3 = e3m + ((size_t)k * ny + j) * nx;
                const float *pv = zv + ((size_t)k * ny + j) * nx;
                const int16_t *pm = ibmask + (size_t)j * nx * nb + b;
                for (int i = 0; i < nx; ++i) {
                    float t = pe1[i] * pe3[i];
                    t = t * (float)pm[(size_t)i * nb];
                    t = t * pv[i];
                    acc = acc - (double)t;
                }
                dmoc[((size_t)k * ny + j) * nb + b] = acc;
            }
        }
#pragma omp parallel for schedule(runtime)
    for (int j = 0; j < ny; ++j)
        for (int k = nz - 2; k >= 0; --k)
            for (int b = 0; b < nb; ++b) {
                size_t o = ((size_t)k * ny + j) * nb + b;
                size_t o1 = ((size_t)(k + 1) * ny + j) * nb + b;
                dmoc[o] = dmoc[o1] + dmoc[o] / 1.0e6;
            }
}

/* a5. output conversion -- src/cdfmoc.f90:520-551.  out has (nb + (nb>=5)) variables of (nz,ny) REAL(4):
 * out[v][k][j] = REAL(dmoc(v,j,k)); last variable inp0 = REAL(dmoc(glo)-dmoc(atl)) (:549). */
void oracle_cdfmoc_output(int ny, int nz, int nb, const double *dmoc, float *out)
{
    for (int b = 0; b < nb; ++b)
        for (int k = 0; k < nz; ++k)
            for (int j = 0; j < ny; ++j)
                out[((size_t)b * nz + k) * ny + j] = (float)dmoc[((size_t)k * ny + j) * nb + b];
    if (nb >= 5)
        for (int k = 0; k < nz; ++k)
            for (int j = 0; j < ny; ++j) {
                size_t o = ((size_t)k * ny + j) * nb;
                out[((size_t)nb * nz + k) * ny + j] = (float)(dmoc[o + 0] - dmoc[o + 1]);
            }
}

/* ---------------------------------------------------------------------------------------------
 * a8. sigmai_dep -- src/eos.f90:842-882 (coefficients: eos_init :207-279 / :408-466).
 * `teos10` selects the coefficient set.  pref is REAL(4) widened before dlh = pref*r1_Z0.
 * eos_dlr() is the four nested Horner polynomials and their combination (:858-879), parenthesised
 * exactly as the reference writes them.
 * ------------------------------------------------------------------------------------------- */
static inline double eos_dlr(const double *C, double dlt, double dls, double dlh)
{
#define E(i, j, k) C[I_EOS##i##j##k]
    double dlr3 = E(0, 1, 3) * dlt + E(1, 0, 3) * dls + E(0, 0, 3);
    double dlr2 = (E(0, 2, 2) * dlt + E(1, 1, 2) * dls + E(0, 1, 2)) * dlt + (E(2, 0, 2) * dls + E(1, 0, 2)) * dls +
                  E(0, 0, 2);
    double dlr1 = (((E(0, 4, 1) * dlt + E(1, 3, 1) * dls + E(0, 3, 1)) * dlt + (E(2, 2, 1) * dls + E(1, 2, 1)) * dls +
                    E(0, 2, 1)) * dlt +
                   ((E(3, 1, 1) * dls + E(2, 1, 1)) * dls + E(1, 1, 1)) * dls + E(0, 1, 1)) * dlt +
                  (((E(4, 0, 1) * dls + E(3, 0, 1)) * dls + E(2, 0, 1)) * dls + E(1, 0, 1)) * dls + E(0, 0, 1);
    double dlr0 =
        (((((E(0, 6, 0) * dlt + E(1, 5, 0) * dls + E(0, 5, 0)) * dlt + (E(2, 4, 0) * dls + E(1, 4, 0)) * dls +
            E(0, 4, 0)) * dlt +
           ((E(3, 3, 0) * dls + E(2, 3, 0)) * dls + E(1, 3, 0)) * dls + E(0, 3, 0)) * dlt +
          (((E(4, 2, 0) * dls + E(3, 2, 0)) * dls + E(2, 2, 0)) * dls + E(1, 2, 0)) * dls + E(0, 2, 0)) * dlt +
         ((((E(5, 1, 0) * dls + E(4, 1, 0)) * dls + E(3, 1, 0)) * dls + E(2, 1, 0)) * dls + E(1, 1, 0)) * dls +
         E(0, 1, 0)) * dlt +
        (((((E(6, 0, 0) * dls + E(5, 0, 0)) * dls + E(4, 0, 0)) * dls + E(3, 0, 0)) * dls + E(2, 0, 0)) * dls +
         E(1, 0, 0)) * dls +
        E(0, 0, 0);
#undef E
    return ((dlr3 * dlh + dlr2) * dlh + dlr1) * dlh + dlr0;
}

void oracle_sigmai_dep(size_t n, const float *ptem, const float *psal, float pref, int teos10, double *out)
{
    const double *C = teos10 ? CDF_TEOS10_COEF : CDF_EOS80_COEF;
    const double rdeltaS = teos10 ? CDF_TEOS10_RDELTAS : CDF_EOS80_RDELTAS;
    const double r1_S0 = teos10 ? CDF_TEOS10_R1_S0 : CDF_EOS80_R1_S0;
    const double r1_T0 = 1.0 / 40.0;
    const double r1_Z0 = 1.e-4;
    const double rau0 = 1000.0;
    const double *R = CDF_EOS_R0;
    double dlh = (double)pref * r1_Z0;
    double dlref = (((((R[5] * dlh + R[4]) * dlh + R[3]) * dlh + R[2]) * dlh + R[1]) * dlh + R[0]) * dlh;
#pragma omp parallel for schedule(static)
    for (size_t c = 0; c < n; ++c) {
        double dlt = (double)ptem[c] * r1_T0;
        double dls = sqrt(fabs((double)psal[c] + rdeltaS) * r1_S0);
        double dltm = (psal[c] == 0.0f) ? 0.0 : 1.0;
        double dlr = eos_dlr(C, dlt, dls, dlh);
        out[c] = (dlr + dlref - rau0) * dltm;
    }
}

/* dlr alone: the quantity the reference's comment check values are quoted on (eos.f90:817,820 vs :879). */
double oracle_eos_dlr(float t, float s, float depth, int teos10)
{
    const double *C = teos10 ? CDF_TEOS10_COEF : CDF_EOS80_COEF;
    const double rdeltaS = teos10 ? CDF_TEOS10_RDELTAS : CDF_EOS80_RDELTAS;
    const double r1_S0 = teos10 ? CDF_TEOS10_R1_S0 : CDF_EOS80_R1_S0;
    double dlt = (double)t * (1.0 / 40.0);
    double dls = sqrt(fabs((double)s + rdeltaS) * r1_S0);
    return eos_dlr(C, dlt, dls, (double)depth * 1.e-4);
}

/* sigmantr -- src/eos.f90:661-684 (McDougall & Jackett 2005 neutral density, minus 1000). */
void oracle_sigmantr(size_t n, const float *ptem, const float *psal, double *out)
{
#pragma omp parallel for schedule(static)
    for (size_t c = 0; c < n; ++c) {
        double dl_t = ptem[c];
        double dl_s = psal[c];
        double dl_sr = sqrt(fabs(dl_s));
        double dl_r1 = ((-4.3159255086706703e-4 * dl_t + 8.1157118782170051e-2) * dl_t + 2.2280832068441331e-1) * dl_t +
                       1002.3063688892480e0;
        double dl_r2 = (-1.7052298331414675e-7 * dl_s - 3.1710675488863952e-3 * dl_t - 1.0304537539692924e-4) * dl_s;
        double dl_r3 = (((-2.3850178558212048e-9 * dl_t - 1.6212552470310961e-7) * dl_t + 7.8717799560577725e-5) * dl_t +
                        4.3907692647825900e-5) * dl_t + 1.0e0;
        double dl_r4 = ((-2.2744455733317707e-9 * dl_t * dl_t + 6.0399864718597388e-6) * dl_t - 5.1268124398160734e-4) * dl_s;
        double dl_r5 = (-1.3409379420216683e-9 * dl_t * dl_t - 3.6138532339703262e-5) * dl_s * dl_sr;
        out[c] = (dl_r1 + dl_r2) / (dl_r3 + dl_r4 + dl_r5) - 1000.e0;
    }
}

/* a12. bin axis -- src/cdfmocsig.f90:302-304: sigma(ji) = sigmin + (ji-0.5)*sigstp, all REAL(4). */
void oracle_sigma_axis(int nbins, float sigmin, float sigstp, float *sigma)
{
    for (int n = 1; n <= nbins; ++n) {
        float t = (float)n - 0.5f;
        t = t * sigstp;
        sigma[n - 1] = sigmin + t;
    }
}

/* a12. default bins by INT(pref) -- src/cdfmocsig.f90:265-292.  returns 0 ok, 99 = STOP 99. */
int oracle_default_bins(float pref, int lntr, int *nbins, float *sigmin, float *sigstp)
{
    if (lntr) { *nbins = 52; *sigmin = 1023.f; *sigstp = 0.1f; return 0; }
    switch ((int)pref) {
    case 0: *nbins = 52; *sigmin = 23.f; *sigstp = 0.1f; return 0;
    case 1000: *nbins = 88; *sigmin = 24.f; *sigstp = 0.1f; return 0;
    case 2000: *nbins = 158; *sigmin = 30.f; *sigstp = 0.05f; return 0;
    default: return 99;
    }
}

/* ---------------------------------------------------------------------------------------------
 * a6..a9 for one level: scrub, area, itmask, density, bin -- src/cdfmocsig.f90:374-403.
 * zv/zt/zs are scrubbed IN PLACE (as the WHERE statements do); zarea, ibin are outputs.
 * eos: 0 EOS80, 1 TEOS10, 2 neutral (-ntr).
 * ------------------------------------------------------------------------------------------- */
void oracle_mocsig_level_prep(int nx, int ny, float *zv, float *zt, float *zs, const float *zveiv, const float *e1v,
                              const float *e3v, float zspv, float zspt, float zsps, float pref, int eos, float sigmin,
                              float sigstp, int nbins, float *zarea, int16_t *itmask, int32_t *ibin, double *dens)
{
    size_t n = (size_t)nx * ny;
    for (size_t c = 0; c < n; ++c)
        if (zv[c] == zspv) zv[c] = 0.f; /* :375 */
    if (zveiv)
        for (size_t c = 0; c < n; ++c) zv[c] = zv[c] + zveiv[c]; /* :378 */
    for (size_t c = 0; c < n; ++c)
        if (zt[c] == zspt) zt[c] = 0.f; /* :383 */
    for (size_t c = 0; c < n; ++c)
        if (zs[c] == zsps) zs[c] = 0.f; /* :384 */
    for (size_t c = 0; c < n; ++c) zarea[c] = e1v[c] * e3v[c]; /* :390, e3v NOT vmask-masked */
    for (size_t c = 0; c < n; ++c) itmask[c] = (zs[c] == zsps) ? 0 : 1; /* :393-394 (after the scrub) */
    if (eos == CDF_EOS_NEUTRAL)
        oracle_sigmantr(n, zt, zs, dens); /* :395 */
    else
        oracle_sigmai_dep(n, zt, zs, pref, eos == CDF_EOS_TEOS10, dens); /* :396 */
    for (size_t c = 0; c < n; ++c) {
        float zttmp = (float)(dens[c] * (double)itmask[c]); /* :399 */
        float q = (zttmp - sigmin) / sigstp;                 /* :401 REAL(4) */
        int32_t ib = (int32_t)q;                             /* INT() truncates toward zero */
        if (ib < 1) ib = 1;                                  /* :402 */
        if (ib > nbins) ib = nbins;                          /* :403 */
        ibin[c] = ib;
    }
}

/* ---------------------------------------------------------------------------------------------
 * a10 faithful: src/cdfmocsig.f90:405-442 -- dmoc_tmp(nbins,nx) zeroed per row, scatter, then the
 * DENSE (basin, bin, i) accumulation with dmoc_tmp*ibmask in REAL(8).
 * a10 direct: the same sums without the dense pass (adds only the non-zero entry of each column).
 * Adding +0.0 to an accumulator that started at +0.0 never changes it, so both forms are bit-identical
 * for finite inputs; the direct form is what an O(cells) CPU code would do and is the fair baseline.
 * ------------------------------------------------------------------------------------------- */
void oracle_mocsig_level_accum(int nx, int ny, int nb, int nbins, const float *zv, const float *zarea,
                               const int32_t *ibin, const int16_t *ibmask, int faithful, double *dmoc)
{
    int ij1 = 1, ij2 = ny - 2; /* 0-based jj=2..npjglo-1 */
    if (ny <= 1) { ij1 = 0; ij2 = 0; }
#pragma omp parallel
    {
        double *tmp = faithful ? (double *)malloc(sizeof(double) * (size_t)nbins * nx) : NULL;
#pragma omp for schedule(runtime)
        for (int j = ij1; j <= ij2; ++j) {
            if (faithful) {
                memset(tmp, 0, sizeof(double) * (size_t)nbins * nx);
                for (int i = 1; i <= nx - 2; ++i) {
                    size_t c = (size_t)j * nx + i;
                    int ib = ibin[c] - 1;
                    float p = zv[c] * zarea[c];
                    tmp[(size_t)i * nbins + ib] = tmp[(size_t)i * nbins + ib] - (double)p;
                }
                for (int b = 0; b < nb; ++b)
                    for (int bin = 0; bin < nbins; ++bin) {
                        double acc = dmoc[((size_t)j * nbins + bin) * nb + b];
                        for (int i = 1; i <= nx - 2; ++i)
                            acc = acc + tmp[(size_t)i * nbins + bin] * (double)ibmask[((size_t)j * nx + i) * nb + b];
                        dmoc[((size_t)j * nbins + bin) * nb + b] = acc;
                    }
            } else {
                for (int i = 1; i <= nx - 2; ++i) {
                    size_t c = (size_t)j * nx + i;
                    int ib = ibin[c] - 1;
                    float p = zv[c] * zarea[c];
                    double t = 0.0 - (double)p;
                    for (int b = 0; b < nb; ++b)
                        dmoc[((size_t)j * nbins + ib) * nb + b] += t * (double)ibmask[c * nb + b];
                }
            }
        }
        free(tmp);
    }
}

/* a11. bin cumsum -- src/cdfmocsig.f90:471-475 (1.e6 is REAL(4), exactly 10^6). */
void oracle_mocsig_cumsum(int ny, int nb, int nbins, double *dmoc)
{
    for (int j = 0; j < ny; ++j)
        for (int b = 0; b < nb; ++b) dmoc[((size_t)j * nbins + (nbins - 1)) * nb + b] /= 1.0e6;
    for (int bin = nbins - 2; bin >= 0; --bin)
        for (int j = 0; j < ny; ++j)
            for (int b = 0; b < nb; ++b) {
                size_t o = ((size_t)j * nbins + bin) * nb + b;
                size_t o1 = ((size_t)j * nbins + bin + 1) * nb + b;
                dmoc[o] = dmoc[o1] + dmoc[o] / 1.0e6;
            }
}

/* Whole cdfmocsig record -- src/cdfmocsig.f90:366-475.
 * zv,zt,zs: raw file values for levels 1..nz-1, (nz-1,ny,nx); e3v: UNmasked (nz,ny,nx) (or per record with -vvl).
 * zveiv may be NULL.  ibin_out (optional, (nz-1,ny,nx) int32) receives the bin of every cell for bit-exact checks. */
void oracle_cdfmocsig_record(int nx, int ny, int nz, int nb, int nbins, float sigmin, float sigstp, float pref, int eos,
                             const float *e1v, const float *e3v, const int16_t *ibmask, float zspv, float zspt,
                             float zsps, const float *zv_in, const float *zt_in, const float *zs_in,
                             const float *zveiv_in, int faithful, double *dmoc, int32_t *ibin_out)
{
    size_t n = (size_t)nx * ny;
    float *zv = malloc(4 * n), *zt = malloc(4 * n), *zs = malloc(4 * n), *zarea = malloc(4 * n);
    int16_t *itmask = malloc(2 * n);
    int32_t *ibin = malloc(4 * n);
    double *dens = malloc(8 * n);
    memset(dmoc, 0, sizeof(double) * (size_t)nb * nbins * ny);
    for (int k = 0; k < nz - 1; ++k) {
        memcpy(zv, zv_in + k * n, 4 * n);
        memcpy(zt, zt_in + k * n, 4 * n);
        memcpy(zs, zs_in + k * n, 4 * n);
        oracle_mocsig_level_prep(nx, ny, zv, zt, zs, zveiv_in ? zveiv_in + k * n : NULL, e1v, e3v + k * n, zspv, zspt,
                                 zsps, pref, eos, sigmin, sigstp, nbins, zarea, itmask, ibin, dens);
        if (ibin_out) memcpy(ibin_out + k * n, ibin, 4 * n);
        oracle_mocsig_level_accum(nx, ny, nb, nbins, zv, zarea, ibin, ibmask, faithful, dmoc);
    }
    oracle_mocsig_cumsum(ny, nb, nbins, dmoc);
    free(zv); free(zt); free(zs); free(zarea); free(itmask); free(ibin); free(dens);
}

/* output conversion -- src/cdfmocsig.f90:478-483: out[b][bin][j] = REAL(dmoc(b,bin,j)); no inp0. */
void oracle_cdfmocsig_output(int ny, int nb, int nbins, const double *dmoc, float *out)
{
    for (int b = 0; b < nb; ++b)
        for (int bin = 0; bin < nbins; ++bin)
            for (int j = 0; j < ny; ++j)
                out[((size_t)b * nbins + bin) * ny + j] = (float)dmoc[((size_t)j * nbins + bin) * nb + b];
}

/* cdfmaxmoc -- src/cdfmaxmoc.f90:158-167: MAXVAL/MINVAL/MAXLOC/MINLOC of rmoc(1,ijmin:ijmax,ikmin:ikmax), REAL(4)
 * values as read from moc.nc; first occurrence in array order (jj fastest).  Indices 1-based inclusive.
 * NaN cells are skipped as gfortran's intrinsics skip them: a window whose cells are all NaN gives NaN and its first
 * cell; otherwise the first cell holding the extremum, also when that is -Inf (max) or +Inf (min).
 * rmoc[k][j] float32.  out: ovt[2] = max,min ; loc[4] = jj,jk of max, jj,jk of min. */
void oracle_maxmoc(int ny, const float *rmoc, int ijmin, int ijmax, int ikmin, int ikmax, float *ovt, int *loc)
{
    float vmax = NAN, vmin = NAN;
    int seen = 0;
    loc[0] = loc[2] = ijmin; loc[1] = loc[3] = ikmin;
    for (int k = ikmin; k <= ikmax; ++k)
        for (int j = ijmin; j <= ijmax; ++j) {
            const float v = rmoc[(size_t)(k - 1) * ny + (j - 1)];
            if (isnan(v)) continue;
            if (!seen || v > vmax) { vmax = v; loc[0] = j; loc[1] = k; }
            if (!seen || v < vmin) { vmin = v; loc[2] = j; loc[3] = k; }
            seen = 1;
        }
    ovt[0] = vmax; ovt[1] = vmin;
}

/* -isodep -- src/cdfmocsig.f90:423-430,444-454,463-469: zonal-mean depth of the isopycnals.
 *   depi_tmp(ib,ji) += gdep(jk) * itmask(ji,jj) * zarea(ji,jj)      (REAL(4) chain, added into REAL(8))
 *   wdep_tmp(ib,ji) +=            itmask(ji,jj) * zarea(ji,jj)
 *   depi(b,bin,jj)  += depi_tmp(bin,ji) * ibmask(b,ji,jj) ; same for wdep ; i = 2..nx-1, j = 2..ny-1
 * One level: accumulates into depi/wdep (ny,nbins,nb).  gdepk = -gdept(jk) (cdfmocsig.f90:328). */
void oracle_isodep_level_accum(int nx, int ny, int nb, int nbins, float gdepk, const float *zarea, const int16_t *itmask,
                               const int32_t *ibin, const int16_t *ibmask, double *depi, double *wdep)
{
    int ij1 = 1, ij2 = ny - 2;
    if (ny <= 1) { ij1 = 0; ij2 = 0; }
    for (int j = ij1; j <= ij2; ++j)
        for (int i = 1; i <= nx - 2; ++i) {
            size_t c = (size_t)j * nx + i;
            int ib = ibin[c] - 1;
            float a = gdepk * (float)itmask[c];
            a = a * zarea[c];
            float w = (float)itmask[c] * zarea[c];
            for (int b = 0; b < nb; ++b) {
                size_t o = ((size_t)j * nbins + ib) * nb + b;
                depi[o] += (double)a * (double)ibmask[c * nb + b];
                wdep[o] += (double)w * (double)ibmask[c * nb + b];
            }
        }
}

/* Whole record with -isodep: returns both the MOC (as oracle_cdfmocsig_record) and depi (ny,nbins,nb), already
 * divided by wdep where wdep /= 0 and set to 99999. elsewhere (cdfmocsig.f90:463-469). */
void oracle_cdfmocsig_record_isodep(int nx, int ny, int nz, int nb, int nbins, float sigmin, float sigstp, float pref,
                                    int eos, const float *e1v, const float *e3v, const int16_t *ibmask, float zspv,
                                    float zspt, float zsps, const float *gdept, const float *zv_in, const float *zt_in,
                                    const float *zs_in, double *dmoc, double *depi)
{
    size_t n = (size_t)nx * ny;
    float *zv = malloc(4 * n), *zt = malloc(4 * n), *zs = malloc(4 * n), *zarea = malloc(4 * n);
    int16_t *itmask = malloc(2 * n);
    int32_t *ibin = malloc(4 * n);
    double *dens = malloc(8 * n);
    size_t no = (size_t)nb * nbins * ny;
    double *wdep = calloc(no, 8);
    memset(dmoc, 0, 8 * no);
    memset(depi, 0, 8 * no);
    for (int k = 0; k < nz - 1; ++k) {
        memcpy(zv, zv_in + k * n, 4 * n);
        memcpy(zt, zt_in + k * n, 4 * n);
        memcpy(zs, zs_in + k * n, 4 * n);
        oracle_mocsig_level_prep(nx, ny, zv, zt, zs, NULL, e1v, e3v + k * n, zspv, zspt, zsps, pref, eos, sigmin, sigstp,
                                 nbins, zarea, itmask, ibin, dens);
        oracle_mocsig_level_accum(nx, ny, nb, nbins, zv, zarea, ibin, ibmask, 0, dmoc);
        oracle_isodep_level_accum(nx, ny, nb, nbins, -gdept[k], zarea, itmask, ibin, ibmask, depi, wdep);
    }
    for (size_t o = 0; o < no; ++o) depi[o] = (wdep[o] != 0.0) ? depi[o] / wdep[o] : 99999.0;
    oracle_mocsig_cumsum(ny, nb, nbins, dmoc);
    free(zv); free(zt); free(zs); free(zarea); free(itmask); free(ibin); free(dens); free(wdep);
}

/* ---------------------------------------------------------------------------------------------
 * cdfmoc -decomp -- src/cdfmoc.f90:353,360-365,390-517 (SURVEY.md App. E.1).  One time record.
 * Types as declared in the reference (:101-117): hdep, zcoef, zsig0, zmsv, zv REAL(4); dvbt, dvgeo, dgeo and all
 * dmoc_* REAL(8).  Inputs: e3m = e3v*vmask (nz,ny,nx); umask, tmask (nz,ny,nx) INTEGER(2); zv, zt, zs levels 1..nz-1;
 * gphiv (ny,nx); gdept (nz).  dmoc_sh is IN/OUT: the reference never zeroes it (:299,:471) -- pass zeros for npt=1.
 * Outputs (nz,ny,nb): dmoc (total), dmoc_sh, dmoc_bt, dmoc_ag.  Level nz of every array is left as given/zero.
 * ------------------------------------------------------------------------------------------- */
static void zonal_weighted(int nx, int ny, int nz, int nb, const float *e1v, const float *e3m, const int16_t *ibmask,
                           const double *dvbt, double *out)
{   /* :403-415 / :490-502: out(b,jj,jk) -= e1v*e3v*ibmask*dvbt  (REAL(4) triple product, REAL(8) last multiply) */
    for (int k = 0; k < nz - 1; ++k)
        for (int j = 0; j < ny; ++j)
            for (int b = 0; b < nb; ++b) {
                double acc = out[((size_t)k * ny + j) * nb + b];
                for (int i = 0; i < nx; ++i) {
                    size_t c = (size_t)j * nx + i;
                    float t = e1v[c] * e3m[(size_t)k * ny * nx + c];
                    t = t * (float)ibmask[c * nb + b];
                    acc = acc - (double)t * dvbt[c];
                }
                out[((size_t)k * ny + j) * nb + b] = acc;
            }
}

void oracle_cdfmoc_decomp_record(int nx, int ny, int nz, int nb, int teos10, const float *e1v, const float *e1u,
                                 const float *gphiv, const float *gdept, const float *e3m, const int16_t *ibmask,
                                 const int16_t *umask, const int16_t *tmask, const float *zv_in, const float *zt_in,
                                 const float *zs_in, double *dmoc, double *dmoc_sh, double *dmoc_bt, double *dmoc_ag)
{
    const size_t nxy = (size_t)nx * ny, nout = (size_t)nb * ny * nz;
    double *dvbt = calloc(nxy, 8), *dvgeo = calloc(2 * nxy, 8), *dmoc_btw = calloc(nout, 8), *dens = malloc(8 * nxy);
    float *hdep = calloc(nxy, 4), *zcoef = malloc(4 * nxy), *zsig0 = malloc(4 * nxy), *zv = malloc(4 * nxy);
    /* 1) total MOC + barotropic sums (:352-388, :360-365) */
    oracle_cdfmoc_record(nx, ny, nz, nb, e1v, e3m, ibmask, zv_in, dmoc);
    for (int k = 0; k < nz - 1; ++k)
        for (size_t c = 0; c < nxy; ++c) {
            float t = e3m[k * nxy + c] * zv_in[k * nxy + c];
            dvbt[c] = dvbt[c] + (double)t;              /* dvbt + e3v*zv*1.d0 */
            hdep[c] = hdep[c] + e3m[k * nxy + c];       /* REAL(4) running sum */
        }
    memcpy(zv, zv_in + (size_t)(nz - 2) * nxy, 4 * nxy);   /* zv keeps the last level read (:357) */
    /* 2.1) barotropic (:397-419) */
    for (size_t c = 0; c < nxy; ++c) dvbt[c] = (hdep[c] != 0.f) ? dvbt[c] / (double)hdep[c] : 0.0;
    memset(dmoc_bt, 0, 8 * nout);
    zonal_weighted(nx, ny, nz, nb, e1v, e3m, ibmask, dvbt, dmoc_bt);
    for (int k = nz - 2; k >= 0; --k)
        for (size_t o = 0; o < (size_t)ny * nb; ++o)
            dmoc_bt[(size_t)k * ny * nb + o] = dmoc_bt[(size_t)(k + 1) * ny * nb + o] + dmoc_bt[(size_t)k * ny * nb + o] / 1.0e6;
    /* 2.2) geostrophic shear (:425-478) */
    {
        const float rau0 = 1025.0f, grav = 9.81f;
        const float rpi = acosf(-1.f);
        for (size_t c = 0; c < nxy; ++c) {
            float f = 2 * 2 * rpi;                      /* 2*2*rpi/(24.0*3600.)*SIN(rpi*gphiv/180.0), left to right */
            f = f / (24.0f * 3600.f);
            float a = rpi * gphiv[c];
            a = a / 180.0f;
            f = f * sinf(a);
            if (f != 0.f) { float g = -grav / rau0; zcoef[c] = g / f; } else zcoef[c] = 0.f;
        }
    }
    memset(dvbt, 0, 8 * nxy);
    int iup = 0, ido = 1;
    for (int k = nz - 2; k >= 0; --k) {
        const int16_t *um = umask + k * nxy, *tm = tmask + k * nxy;
        oracle_sigmai_dep(nxy, zt_in + k * nxy, zs_in + k * nxy, gdept[k], teos10, dens);
        for (size_t c = 0; c < nxy; ++c) zsig0[c] = (float)(dens[c] * (double)tm[c]);
        for (int j = 1; j <= ny - 2; ++j)
            for (int i = 1; i <= nx - 2; ++i) {
                size_t c = (size_t)j * nx + i, cn = c + nx;   /* (ji,jj) and (ji,jj+1) */
                int16_t su = (int16_t)(um[cn - 1] + um[cn] + um[c - 1] + um[c]);
                float zmsv = 1.f / (float)(su > 1 ? su : 1);
                float t1 = (zsig0[cn] - zsig0[cn - 1]) * (float)um[cn - 1]; t1 = t1 / e1u[cn - 1];
                float t2 = (zsig0[cn + 1] - zsig0[cn]) * (float)um[cn];     t2 = t2 / e1u[cn];
                float t3 = (zsig0[c] - zsig0[c - 1]) * (float)um[c - 1];    t3 = t3 / e1u[c - 1];
                float t4 = (zsig0[c + 1] - zsig0[c]) * (float)um[c];        t4 = t4 / e1u[c];
                float sgeo = t1 + t2; sgeo = sgeo + t3; sgeo = sgeo + t4;
                double dgeo = (double)sgeo;
                double d = (double)zcoef[c] * dgeo;
                d = d * (double)zmsv;
                d = d * (double)ibmask[c * nb + 0];
                d = d * (double)e3m[k * nxy + c];
                dvgeo[iup * nxy + c] = dvgeo[ido * nxy + c] + d;
                zv[c] = (float)(0.5 * (dvgeo[iup * nxy + c] + dvgeo[ido * nxy + c]));
            }
        for (size_t c = 0; c < nxy; ++c) {
            float t = e3m[k * nxy + c] * zv[c];
            dvbt[c] = dvbt[c] + (double)t;
        }
        for (int j = 0; j < ny; ++j)
            for (int b = 0; b < nb; ++b) {
                double acc = dmoc_sh[((size_t)k * ny + j) * nb + b];
                for (int i = 0; i < nx; ++i) {
                    size_t c = (size_t)j * nx + i;
                    float t = e1v[c] * e3m[k * nxy + c];
                    t = t * (float)ibmask[c * nb + b];
                    t = t * zv[c];
                    acc = acc - (double)t;
                }
                dmoc_sh[((size_t)k * ny + j) * nb + b] = acc;
            }
        int tmp = iup; iup = ido; ido = tmp;
    }
    for (size_t c = 0; c < nxy; ++c) dvbt[c] = (hdep[c] != 0.f) ? dvbt[c] / (double)hdep[c] : 0.0;
    /* 2.2.1) pseudo-barotropic part of the shear (:489-505) */
    zonal_weighted(nx, ny, nz, nb, e1v, e3m, ibmask, dvbt, dmoc_btw);
    for (size_t o = 0; o < nout; ++o) dmoc_sh[o] = dmoc_sh[o] - dmoc_btw[o];
    for (int k = nz - 2; k >= 0; --k)
        for (size_t o = 0; o < (size_t)ny * nb; ++o)
            dmoc_sh[(size_t)k * ny * nb + o] = dmoc_sh[(size_t)(k + 1) * ny * nb + o] + dmoc_sh[(size_t)k * ny * nb + o] / 1.0e6;
    /* 2.3) ageostrophic (:516) */
    for (size_t o = 0; o < nout; ++o) dmoc_ag[o] = dmoc[o] - dmoc_sh[o] - dmoc_bt[o];
    free(dvbt); free(dvgeo); free(dmoc_btw); free(dens); free(hdep); free(zcoef); free(zsig0); free(zv);
}

/* zcoef of :428-433 alone (the host computes it with libm's sinf, exactly as the Fortran run-time does) */
void oracle_decomp_zcoef(size_t n, const float *gphiv, float *zcoef)
{
    const float rau0 = 1025.0f, grav = 9.81f;
    const float rpi = acosf(-1.f);
    for (size_t c = 0; c < n; ++c) {
        float f = 2 * 2 * rpi;
        f = f / (24.0f * 3600.f);
        float a = rpi * gphiv[c];
        a = a / 180.0f;
        f = f * sinf(a);
        if (f != 0.f) { float g = -grav / rau0; zcoef[c] = g / f; } else zcoef[c] = 0.f;
    }
}

/* =============================================================================================
 * Sibling tools (SURVEY.md section 8 f3): the same masked zonal integral behind other command lines.
 * PARITY UNPINNED by the reference (no tests / golden vectors); pinned by the NumPy restatements in
 * oracle/np_oracle.py and by property tests.
 * ============================================================================================= */

/* zonal basin masks of cdfzonalsum / cdfzonalmean -- src/cdfzonalsum.f90:286-296, cdfzonalmean.f90:287-297.
 * REAL(4) planes: 1 global (the variable's mask at level 1), 2 atl, 4 ind, 5 pac, 3 = ind + pac clipped to 1.
 * zmask(npbasins,npiglo,npjglo) -> zmask[(j*nx+i)*nb+b]; NO zeroing of the i=1 / i=nx columns here. */
void oracle_zonal_masks(int nx, int ny, int nb, const float *msk1, const float *atl, const float *ind, const float *pac,
                        float *zmask)
{
    for (size_t c = 0; c < (size_t)nx * ny; ++c) {
        zmask[c * nb + 0] = msk1[c];
        if (nb == 5) {
            zmask[c * nb + 1] = atl[c];
            zmask[c * nb + 3] = ind[c];
            zmask[c * nb + 4] = pac[c];
            float z = pac[c] + ind[c];
            if (z > 0.0f) z = 1.0f;
            zmask[c * nb + 2] = z;
        }
    }
}

/* dl_surf(:,:) = 1.d0 * e1(:,:) * e2(:,:) -- cdfzonalsum.f90:257, cdfzonalmean.f90:265: (1.d0*e1)*e2 in REAL(8) */
void oracle_zonal_dlsurf(size_t n, const float *e1, const float *e2, double *dl)
{
    for (size_t c = 0; c < n; ++c) dl[c] = (1.0 * (double)e1[c]) * (double)e2[c];
}

/* cdfzonalsum, one level -- src/cdfzonalsum.f90:309-322.
 *   dtmp = zmask(jbasin,ji,jj)*zmaskvar(ji,jj)*zv(ji,jj)*1.d0   : REAL(4) products left to right, then REAL(8)
 *   dzosum(jj,jk) = dzosum(jj,jk) + dl_surf(ji,jj)*dtmp ; dzosum(:,jk) = dzosum(:,jk) / alpha(:)  (alpha REAL(4))
 * out[b*ny + j] */
void oracle_zonalsum_level(int nx, int ny, int nb, const float *zmask, const float *zmaskvar, const float *zv,
                           const double *dl_surf, const float *alpha, double *out)
{
#pragma omp parallel for schedule(static)
    for (int j = 0; j < ny; ++j)
        for (int b = 0; b < nb; ++b) {
            double acc = 0.0;
            for (int i = 0; i < nx; ++i) {
                const size_t c = (size_t)j * nx + i;
                const float p1 = zmask[c * nb + b] * zmaskvar[c];
                const float p2 = p1 * zv[c];
                const double dtmp = (double)p2 * 1.0;
                acc = acc + dl_surf[c] * dtmp;
            }
            out[(size_t)b * ny + j] = acc / (double)(alpha ? alpha[j] : 1.0f);
        }
}

/* cdfzonalmean, one level -- src/cdfzonalmean.f90:312-344.
 *   dtmp = 1.d0 * zmask*zmaskvar*zv                  : all REAL(8) (the first operand promotes the chain)
 *   dzomean += dl_surf*dtmp ; darea += dl_surf*zmask*zmaskvar
 *   lmax: rzomax = MAX(rzomax, dtmp) (REAL(4) <- REAL(8)), rzomin = MIN(rzomin, dtmp) where dtmp /= 0 ; start -1.e20 / 1.e20;
 *         a NaN dtmp leaves both unchanged (the reference's MAX / MIN with a NaN depend on the compiler)
 *   mean = dzomean/darea where darea /= 0 else zspval ; rzomax = rzomin = zspval where darea == 0
 * mean[b*ny+j], zmax/zmin[b*ny+j] (may be NULL when lmax == 0) */
void oracle_zonalmean_level(int nx, int ny, int nb, const float *zmask, const float *zmaskvar, const float *zv,
                            const double *dl_surf, float zspval, int lmax, double *mean, float *zmax, float *zmin)
{
#pragma omp parallel for schedule(static)
    for (int j = 0; j < ny; ++j)
        for (int b = 0; b < nb; ++b) {
            double acc = 0.0, area = 0.0;
            float rmax = -1.e20f, rmin = 1.e20f;
            for (int i = 0; i < nx; ++i) {
                const size_t c = (size_t)j * nx + i;
                const double m = (double)zmask[c * nb + b];
                const double dtmp = ((1.0 * m) * (double)zmaskvar[c]) * (double)zv[c];
                acc = acc + dl_surf[c] * dtmp;
                area = area + (dl_surf[c] * m) * (double)zmaskvar[c];
                if (lmax && dtmp == dtmp) {   /* a NaN cell never changes the zonal max / min (include/cdfgpu.h) */
                    const double a = (double)rmax;
                    rmax = (float)(a > dtmp ? a : dtmp);   /* MAX(real4, real8): compared in REAL(8), stored REAL(4) */
                    if (dtmp != 0.0) {
                        const double bb = (double)rmin;
                        rmin = (float)(bb < dtmp ? bb : dtmp);
                    }
                }
            }
            const size_t o = (size_t)b * ny + j;
            mean[o] = (area != 0.0) ? acc / area : (double)zspval;
            if (lmax) {
                zmax[o] = (area == 0.0) ? zspval : rmax;
                zmin[o] = (area == 0.0) ? zspval : rmin;
            }
        }
}

/* cdfmhst, one record (-vt file mode) -- src/cdfmhst.f90:303-366.
 *   dwkh = zvt*e1v*e3v*1.d0 (REAL(4) products, then REAL(8)) ; dtrph += dwkh*pprau0*pprcp (1000., 4000. REAL(4) constants)
 *   dwks likewise ; dtrps += dwks
 *   zonal sums after each level: global SUM(dtrph(2:npiglo-1,jj)*vmask1(2:npiglo-1,jj)); atl / pac / ind over all i.
 * heat, salt: [nlev][4][ny] with nlev = nz (zdim: cumulative after each level) or 1 (after the last level);
 * basin order glo, atl, pac, ind; atl/pac/ind may be NULL (then only glo is written, the others are 0). */
void oracle_mhst_record(int nx, int ny, int nz, const float *e1v, const float *e3v, const float *vmask1, const float *atl,
                        const float *pac, const float *ind, const float *zvt, const float *zvs, int zdim, double *heat,
                        double *salt)
{
    const size_t nxy = (size_t)nx * ny;
    double *dtrph = (double *)calloc(nxy, sizeof(double)), *dtrps = (double *)calloc(nxy, sizeof(double));
    const float *masks[4] = {vmask1, atl, pac, ind};
    const int nlev = zdim ? nz : 1;
    memset(heat, 0, sizeof(double) * nlev * 4 * ny);
    memset(salt, 0, sizeof(double) * nlev * 4 * ny);
    for (int k = 0; k < nz; ++k) {
#pragma omp parallel for schedule(static)
        for (int j = 0; j < ny; ++j)
            for (int i = 0; i < nx; ++i) {
                const size_t c = (size_t)j * nx + i, c3 = (size_t)k * nxy + c;
                const float h1 = zvt[c3] * e1v[c], h2 = h1 * e3v[c3];
                const float s1 = zvs[c3] * e1v[c], s2 = s1 * e3v[c3];
                const double dwkh = (double)h2 * 1.0, dwks = (double)s2 * 1.0;
                dtrph[c] = dtrph[c] + (dwkh * (double)1000.0f) * (double)4000.0f;
                dtrps[c] = dtrps[c] + dwks;
            }
        if (zdim || k == nz - 1) {
            const int lev = zdim ? k : 0;
#pragma omp parallel for schedule(static)
            for (int j = 0; j < ny; ++j)
                for (int m = 0; m < 4; ++m) {
                    if (!masks[m]) continue;
                    const int i0 = (m == 0) ? 1 : 0, i1 = (m == 0) ? nx - 1 : nx;
                    double sh = 0.0, ss = 0.0;
                    for (int i = i0; i < i1; ++i) {
                        const size_t c = (size_t)j * nx + i;
                        sh = sh + dtrph[c] * (double)masks[m][c];
                        ss = ss + dtrps[c] * (double)masks[m][c];
                    }
                    heat[((size_t)lev * 4 + m) * ny + j] = sh;
                    salt[((size_t)lev * 4 + m) * ny + j] = ss;
                }
        }
    }
    free(dtrph);
    free(dtrps);
}

/* ---------------------------------------------------------------------------------------------
 * cdftransig_xy3d -- src/cdftransig_xy3d.f90 (SURVEY.md section 8 f3).
 * Bin axis and look-up table (:229-262): dsigma(nbins) bin centres with an optional refined range from ds1zoom,
 * dsig_edge(nbins+1), and itab(nsigmax) that maps a density counted in steps of ds1scalmin to a bin (1-based; 0 where
 * no bin claims the step).  Returns nsigmax; itab receives min(nsigmax, itab_cap) entries.
 * --------------------------------------------------------------------------------------------- */
int oracle_transig_bins(int nbins, double ds1min, double ds1scal, double ds1zoom, double ds1scalmin_in, double *dsigma,
                        double *dsig_edge, int *itab, int itab_cap)
{
    const double ds1scalmin = ds1scalmin_in < ds1scal ? ds1scalmin_in : ds1scal;   /* :213 MIN(ds1scalmin, ds1scal) */
    int ijtrans = 0;
    for (int ji = 1; ji <= nbins; ++ji) {
        const double dsigtest = ds1min + ((float)ji - 0.5f) * ds1scal;              /* (ji-0.5) is REAL(4), exact */
        if (dsigtest > ds1zoom) {
            if (ijtrans == 0) ijtrans = ji;
            dsigma[ji - 1] = ds1zoom + ((float)(ji - ijtrans) + 0.5f) * ds1scalmin;
        } else
            dsigma[ji - 1] = dsigtest;
    }
    dsig_edge[0] = ds1min;
    for (int ji = 2; ji <= nbins; ++ji) dsig_edge[ji - 1] = 0.5f * (dsigma[ji - 1] + dsigma[ji - 2]);
    dsig_edge[nbins] = dsig_edge[nbins - 1] + ds1scalmin;
    const int nsigmax = (int)lround((dsig_edge[nbins] - dsig_edge[0]) / ds1scalmin);  /* NINT */
    for (int ji = 1; ji <= nsigmax && ji <= itab_cap; ++ji) {
        const double dsigtest = ds1min + ((float)ji - 0.5f) * ds1scalmin;
        int v = 0;
        for (int jj = 1; jj <= nbins; ++jj)
            if (dsigtest > dsig_edge[jj - 1] && dsigtest <= dsig_edge[jj]) v = jj;
        itab[ji - 1] = v;
    }
    return nsigmax;
}

/* INT() of a REAL(8): truncation toward zero; out of range and NaN give INT_MIN (x86 CVTTSD2SI, what gfortran emits) */
static inline int f_int_d(double x)
{
    if (!(x > -2147483649.0 && x < 2147483648.0)) return (int)0x80000000;
    return (int)x;
}

/* One time frame, all levels (:396-453; the reference nests jk outside the frames, the additions into each
 * dusigsig(i,j,bin) then come in another order -- fp64 rounding only).
 *   zmasku / zmaskv: 1 where the frame's zu / zv is not 0 -- recomputed only for the frames of the FIRST tag (:410-415);
 *                    set_masks = 1 stores them (bytes, (nz-1,ny,nx)), 0 uses the stored ones
 *   dens2d = sigmai(zt, zs, pref)  REAL(8)                                                        (:420-424)
 *   zdensu(1:nx-1) = REAL(4)(0.5*(dens(i)+dens(i+1))); zdensu(nx) = zdensu(2) if periodic else 0; *zmasku  (:427-435)
 *   zdensv(:,1:ny-1) likewise in j; row ny is never assigned in the reference (uninitialised): 0 here       (:438-439)
 *   ijb = clamp(INT((zdens - ds1min)/ds1scalmin)+1, 1, nsigmax); ibin = itab(ijb)                            (:442-453)
 *   dusigsig(i,j,ibinu) += dble(fl32(e2u * fl32(zu*e3u))) ; dvsigsig likewise with e1v, zv, e3v            (:454-461)
 * A zero in itab (a step no bin claims) would index dusigsig(:,:,0) in the reference; such cells are skipped here. */
void oracle_transig_record(int nx, int ny, int nzm1, int teos10, float pref, int lperio, double ds1min, double ds1scalmin,
                           int nsigmax, const int *itab, int nbins, const float *e2u, const float *e1v, const float *e3u,
                           const float *e3v, const float *zu, const float *zv, const float *zt, const float *zs,
                           int set_masks, uint8_t *masku, uint8_t *maskv, double *dusigsig, double *dvsigsig)
{
    const size_t nxy = (size_t)nx * ny;
    double *dens = (double *)malloc(nxy * sizeof(double));
    float *zdu = (float *)malloc(nxy * sizeof(float)), *zdv = (float *)malloc(nxy * sizeof(float));
    (void)nbins;
    for (int k = 0; k < nzm1; ++k) {
        const size_t o3 = (size_t)k * nxy;
        oracle_sigmai_dep(nxy, zt + o3, zs + o3, pref, teos10, dens);
        if (set_masks)
            for (size_t c = 0; c < nxy; ++c) {
                masku[o3 + c] = (zu[o3 + c] == 0.0f) ? 0 : 1;
                maskv[o3 + c] = (zv[o3 + c] == 0.0f) ? 0 : 1;
            }
#pragma omp parallel for schedule(static)
        for (int j = 0; j < ny; ++j) {
            for (int i = 0; i < nx - 1; ++i) zdu[(size_t)j * nx + i] = (float)(0.5 * (dens[(size_t)j * nx + i] + dens[(size_t)j * nx + i + 1]));
            zdu[(size_t)j * nx + nx - 1] = (lperio && nx > 2) ? zdu[(size_t)j * nx + 1] : 0.0f;
            for (int i = 0; i < nx; ++i) {
                const size_t c = (size_t)j * nx + i;
                zdu[c] = zdu[c] * (float)masku[o3 + c];
                zdv[c] = (j < ny - 1) ? (float)(0.5 * (dens[c] + dens[c + nx])) : 0.0f;
                zdv[c] = zdv[c] * (float)maskv[o3 + c];
            }
        }
#pragma omp parallel for schedule(static)
        for (int j = 0; j < ny; ++j)
            for (int i = 0; i < nx; ++i) {
                const size_t c = (size_t)j * nx + i;
                int ijb = f_int_d(((double)zdu[c] - ds1min) / ds1scalmin) + 1;
                ijb = ijb < 1 ? 1 : ijb;
                ijb = ijb > nsigmax ? nsigmax : ijb;
                const int bu = itab[ijb - 1];
                ijb = f_int_d(((double)zdv[c] - ds1min) / ds1scalmin) + 1;
                ijb = ijb < 1 ? 1 : ijb;
                ijb = ijb > nsigmax ? nsigmax : ijb;
                const int bv = itab[ijb - 1];
                const float tu = zu[o3 + c] * e3u[o3 + c], tv = zv[o3 + c] * e3v[o3 + c];
                const float pu = e2u[c] * tu, pv = e1v[c] * tv;
                if (bu >= 1) dusigsig[(size_t)(bu - 1) * nxy + c] = dusigsig[(size_t)(bu - 1) * nxy + c] + (double)pu * 1.0;
                if (bv >= 1) dvsigsig[(size_t)(bv - 1) * nxy + c] = dvsigsig[(size_t)(bv - 1) * nxy + c] + (double)pv * 1.0;
            }
    }
    free(dens);
    free(zdu);
    free(zdv);
}

/* ===================================================================================================================
 * cdfsigtrp -- src/cdfsigtrp.f90: density-class transport across a zonal / meridional section (SURVEY.md section 8 f3).
 * Section arrays are (npts, npk) in Fortran = [npk][npts] here.
 * =================================================================================================================== */

/* What the reference does with the section slices it has read, up to the density (:428-460 meridional, :521-555 zonal;
 * the two branches differ only in which file columns are read -- and in one detail: the meridional branch masks the mean
 * temperature (:460), the zonal one does not (:555)).
 *   ddepu(ji,1) = gdept(1); ddepu(ji,jk) = ddepu(ji,jk-1) + MIN(e3w_a, e3w_b)     REAL(8) + REAL(4)     (:428-436 / :521-529)
 *   zu: WHERE (zu == zspu) zu = 0                                                                      (:438-439 / :532-533)
 *   zmask = 0 where either salinity is the missing value; zs = 0.5*(zs_a + zs_b)*zmask  (REAL(4))      (:442-446 / :536-541)
 *   nk = first level whose SUM(zs(:,jk)) is zero (REAL(4) sequential sum)                               (:449-454 / :544-549)
 *   zt = 0.5*(zt_a + zt_b) [* zmask]                                                                    (:458-460 / :553-555)
 * ddepu has npk+1 rows, row 0 = 0 (the reference's ddepu(:,0), zeroed at :402).  Returns nk; the reference leaves nk
 * undefined when no level is all land -- npk is returned then (*found = 0). */
int oracle_sigtrp_prepare(int npts, int npk, int merid, float gdept1, const float *e3w_a, const float *e3w_b, const float *zu_in,
                          float zspu, const float *zs_a, const float *zs_b, float zsps, const float *zt_a, const float *zt_b,
                          double *ddepu, float *zu, float *zs, float *zt, float *zmask, int *found)
{
    for (int i = 0; i < npts; ++i) {
        ddepu[i] = 0.0;
        ddepu[(size_t)npts + i] = (double)gdept1;
    }
    for (int k = 1; k < npk; ++k)
        for (int i = 0; i < npts; ++i) {
            const size_t c = (size_t)k * npts + i;
            const float m = e3w_a[c] < e3w_b[c] ? e3w_a[c] : e3w_b[c]; /* MIN(a,b): b unless a < b */
            ddepu[(size_t)(k + 1) * npts + i] = ddepu[(size_t)k * npts + i] + (double)m;
        }
    for (size_t c = 0; c < (size_t)npk * npts; ++c) {
        zu[c] = (zu_in[c] == zspu) ? 0.0f : zu_in[c];
        zmask[c] = (zs_a[c] == zsps || zs_b[c] == zsps) ? 0.0f : 1.0f;
        float a = zs_a[c] + zs_b[c];
        a = 0.5f * a;
        zs[c] = a * zmask[c];
        float t = zt_a[c] + zt_b[c];
        t = 0.5f * t;
        zt[c] = merid ? t * zmask[c] : t;
    }
    int nk = npk;
    *found = 0;
    for (int k = 0; k < npk; ++k) {
        float s = 0.0f;
        for (int i = 0; i < npts; ++i) s = s + zs[(size_t)k * npts + i];
        if (s == 0.0f) {
            nk = k + 1;
            *found = 1;
            break;
        }
    }
    return nk;
}

/* The compute part of one section (:559-627).
 *   mode 0: dsig = sigmai(zt, zs, refdep)*zmask (sigma0 = sigmai at 0, eos.f90:630); 1: sigmantr*zmask; 2 (-temp): -zt*zmask
 *   dsig(:,0) = dsig(:,1) - 1.e-4 ; land: dsig(jk) = dsig(jk-1) + 1.e-5  (REAL(4) literals, promoted)      (:569-578)
 *   dhiso(ji,jiso): depth where the column's density first reaches dsigma_lev(jiso), linear in ddepu          (:581-601)
 *   dwtrp(ji,jiso): transport from the surface down to dhiso (last box fractional)                            (:604-618)
 *   dwtrpbin = dwtrp(jbin+1) - dwtrp(jbin); dtrpbin(jbin) = SUM over ji                                     (:621-627)
 * gdepw: (npk) REAL(4); ddepw_brk != NULL (-brk): [npk][npts], the column's own w depths (:608).
 * dsig has nk+1 rows (row 0 = the dummy layer); dhiso, dwtrp nbins+1 rows; dwtrpbin nbins rows; any of them may be NULL
 * except dtrpbin. */
void oracle_sigtrp_section(int npts, int npk, int nk, const float *eu, const float *de3, const double *ddepu, const float *gdepw,
                           const float *ddepw_brk, const float *zu, const float *zt, const float *zs, const float *zmask, int mode,
                           float refdep, int teos10, double dsigma_min, double dsigma_max, int nbins, double *dsigma_lev_out,
                           double *dsig_out, double *dhiso_out, double *dwtrp_out, double *dwtrpbin_out, double *dtrpbin)
{
    const size_t n = (size_t)nk * npts;
    double *dsig = (double *)calloc((size_t)(nk + 1) * npts, sizeof(double));
    double *lev = (double *)malloc((size_t)(nbins + 1) * sizeof(double));
    double *dhiso = (double *)malloc((size_t)(nbins + 1) * npts * sizeof(double));
    double *dwtrp = (double *)malloc((size_t)(nbins + 1) * npts * sizeof(double));
    const double dltsig = (dsigma_max - dsigma_min) / nbins;
    lev[0] = dsigma_min;
    for (int c = 2; c <= nbins + 1; ++c) lev[c - 1] = lev[0] + (c - 1) * dltsig; /* :355-359 */
    if (mode == 2) {
        for (size_t c = 0; c < n; ++c) {
            const float m = -zt[c] * zmask[c];
            dsig[npts + c] = (double)m;
        }
    } else {
        if (mode == 1)
            oracle_sigmantr(n, zt, zs, dsig + npts);
        else
            oracle_sigmai_dep(n, zt, zs, refdep, teos10, dsig + npts);
        for (size_t c = 0; c < n; ++c) dsig[npts + c] = dsig[npts + c] * (double)zmask[c];
    }
    for (int i = 0; i < npts; ++i) dsig[i] = dsig[npts + i] - (double)1.e-4f;
    for (int i = 0; i < npts; ++i)
        for (int k = 1; k <= nk; ++k)
            if (zmask[(size_t)(k - 1) * npts + i] == 0.0f) dsig[(size_t)k * npts + i] = dsig[(size_t)(k - 1) * npts + i] + (double)1.e-5f;
#pragma omp parallel for schedule(static)
    for (int iso = 0; iso <= nbins; ++iso) {
        const double dsigma = lev[iso];
        for (int i = 0; i < npts; ++i) {
            double h = ddepu[(size_t)npk * npts + i];
            for (int k = 1; k <= nk; ++k) {
                const double d1 = dsig[(size_t)k * npts + i], d0 = dsig[(size_t)(k - 1) * npts + i];
                if (d1 < dsigma) continue;
                const double dalfa = (dsigma - d0) / (d1 - d0);
                if (fabs(dalfa) > 1.1 || dalfa < 0.0) {
                    h = 0.0;
                } else {
                    const double a = ddepu[(size_t)k * npts + i] * dalfa;
                    const double b = (1.0 - dalfa) * ddepu[(size_t)(k - 1) * npts + i];
                    h = a + b;
                }
                break;
            }
            dhiso[(size_t)iso * npts + i] = h;
            double w = 0.0;
            for (int k = 1; k <= nk - 1; ++k) {
                const float gw1 = ddepw_brk ? ddepw_brk[(size_t)k * npts + i] : gdepw[k];             /* gdepw(jk+1) */
                const float gw0 = ddepw_brk ? ddepw_brk[(size_t)(k - 1) * npts + i] : gdepw[k - 1];   /* gdepw(jk)   */
                const double u = (double)zu[(size_t)(k - 1) * npts + i];
                if ((double)gw1 < h) {
                    const double t = (double)eu[i] * (double)de3[(size_t)(k - 1) * npts + i];
                    w = w + t * u * 1.0;
                } else {
                    const double t = (double)eu[i] * (h - (double)gw0);
                    w = w + t * u * 1.0;
                    break;
                }
            }
            dwtrp[(size_t)iso * npts + i] = w;
        }
    }
    for (int b = 0; b < nbins; ++b) {
        double s = 0.0;
        for (int i = 0; i < npts; ++i) {
            const double d = dwtrp[(size_t)(b + 1) * npts + i] - dwtrp[(size_t)b * npts + i];
            if (dwtrpbin_out) dwtrpbin_out[(size_t)b * npts + i] = d;
            s = s + d;
        }
        dtrpbin[b] = s;
    }
    if (dsigma_lev_out) memcpy(dsigma_lev_out, lev, (size_t)(nbins + 1) * sizeof(double));
    if (dsig_out) memcpy(dsig_out, dsig, (size_t)(nk + 1) * npts * sizeof(double));
    if (dhiso_out) memcpy(dhiso_out, dhiso, (size_t)(nbins + 1) * npts * sizeof(double));
    if (dwtrp_out) memcpy(dwtrp_out, dwtrp, (size_t)(nbins + 1) * npts * sizeof(double));
    free(dsig);
    free(lev);
    free(dhiso);
    free(dwtrp);
}
