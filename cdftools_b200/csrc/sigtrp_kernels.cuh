// sigtrp_kernels.cuh -- K7: cdfsigtrp, transport across a section in density classes.
// Replaces the compute part of one section, src/cdfsigtrp.f90:559-627.  Section arrays are (npts, npk) in the reference
// = [npk][npts] here (the along-section index is the fast one, so consecutive threads read consecutive columns).
//
//   dsig(ji,jk)  = sigmai(zt,zs,refdep)*zmask | sigmantr*zmask | -zt*zmask            (:560-567)  kernel (a), one thread per cell
//   dsig(ji,0)   = dsig(ji,1) - 1.e-4 ; land cells: dsig(jk) = dsig(jk-1) + 1.e-5     (:569-578)  kernel (b), one thread per column
//   dhiso(ji,l)  = depth at which the column first reaches dsigma_lev(l)              (:581-601)  kernel (c), one thread per
//   dwtrp(ji,l)  = transport from the surface down to dhiso(ji,l)                     (:604-618)              (column, level l)
//   dwtrpbin     = dwtrp(l+1) - dwtrp(l) ; dtrpbin(l) = SUM_ji dwtrpbin               (:621-627)  kernel (d), one thread per bin,
//                                                                                                 ji ascending as SUM does
// All fp64 arithmetic is spelled with __dmul_rn / __dadd_rn / __ddiv_rn: no contraction, the reference's association.
// The work is O(npts * nbins * nk) per section (1e6 .. 1e8 operations): latency-bound, not HBM-bound -- the kernels exist
// so that the tool is a drop-in on the same library, they are not a roofline item.
#pragma once
#include "common.cuh"
#include "eos_device.cuh"

namespace cdfgpu {

struct SigtrpParams {
    const float *__restrict__ eu;      // (npts)
    const float *__restrict__ de3;     // (npk, npts)  REAL(8) in the reference, holding REAL(4) file values
    const double *__restrict__ ddepu;  // (npk+1, npts), row 0 = the reference's ddepu(:,0) = 0
    const float *__restrict__ gdepw;   // (npk)
    const float *__restrict__ ddepw;   // (npk, npts) or NULL (-brk: the column's own w depths)
    const float *__restrict__ zu, *__restrict__ zt, *__restrict__ zs, *__restrict__ zmask;   // (npk, npts)
    const double *__restrict__ lev;    // (nbins+1) dsigma_lev
    double *dsig;                      // (nk+1, npts)
    double *dhiso, *dwtrp;             // (nbins+1, npts)
    double *dwtrpbin;                  // (nbins, npts)
    double *dtrpbin;                   // (nbins)
    double dlh, dlref;
    int npts, npk, nk, nbins;
};

// ---- per-cell and per-column arithmetic, shared by the single-section kernels and the batched ones (one column axis of
// `pitch` values per level: npts for one section, the concatenated columns of every section for the batch)

// MODE 0: sigma0 (refdep == 0), 1: sigmai(refdep), 2: neutral density, 3: -temp
template <int MODE>
__device__ __forceinline__ double sigtrp_density(float t, float sal, float zmask, double dlh, double dlref)
{
    if (MODE == 3) return (double)__fmul_rn(-t, zmask);
    // sigma0: dlh = 0 drops the pressure terms exactly -- for finite T, S.  The reference still multiplies them by 0,
    // so an Inf in T or S gives NaN there (Inf * 0), not +-Inf: those cells take the full expression.
    const bool fin = (__float_as_uint(t) & 0x7f800000u) != 0x7f800000u && (__float_as_uint(sal) & 0x7f800000u) != 0x7f800000u;
    const double s = MODE == 2             ? eos_sigma_neutral(t, sal)
                     : (MODE == 0 && fin) ? eos_sigma_exact<true>(t, sal, dlh, dlref)
                                          : eos_sigma_exact<false>(t, sal, dlh, dlref);
    return __dmul_rn(s, (double)zmask);
}

// land fill (:569-578): the top row from the first level, then a land cell (zmask 0) continues its upper neighbour
__device__ __forceinline__ double sigtrp_fill_top(double d1) { return __dadd_rn(d1, -(double)1.e-4f); }
__device__ __forceinline__ double sigtrp_fill_level(double prev, double d, float zmask)
{
    return zmask == 0.0f ? __dadd_rn(prev, (double)1.e-5f) : d;
}

// land fill of one column: dsig rows 0..nk, zmask rows 0..nk-1, consecutive levels `pitch` apart
__device__ __forceinline__ void sigtrp_fill_column(double *dsig, const float *zmask, size_t pitch, int nk)
{
    double prev = sigtrp_fill_top(dsig[pitch]);
    dsig[0] = prev;
    for (int k = 1; k <= nk; ++k) {
        const size_t c = (size_t)k * pitch;
        const float m = zmask[c - pitch];
        const double d = sigtrp_fill_level(prev, dsig[c], m);
        if (m == 0.0f) dsig[c] = d;
        prev = d;
    }
}

// one column and one class limit dsigma (:581-618): h = depth at which the column first reaches dsigma, w = transport from
// the surface down to h.  ddepw: the column's own w depths (-brk) or NULL for gdepw.  FILL: dsig rows 1..nk are not yet
// land-filled; the fill is applied here as the levels are read (zmask rows 0..nk-1), and row 0 is not read.
template <bool FILL>
__device__ __forceinline__ void sigtrp_iso_column(const double *ddepu, const double *dsig, const float *zmask, const float *de3,
                                                  const float *zu, const float *ddepw, const float *gdepw, float eu, double dsigma,
                                                  size_t pitch, int npk, int nk, double &h_out, double &w_out)
{
    double h = ddepu[(size_t)npk * pitch];
    double d0 = FILL ? sigtrp_fill_top(dsig[pitch]) : dsig[0];
    for (int k = 1; k <= nk; ++k) {
        double d1 = dsig[(size_t)k * pitch];
        if (FILL) d1 = sigtrp_fill_level(d0, d1, zmask[(size_t)(k - 1) * pitch]);
        if (!(d1 < dsigma)) {
            const double dalfa = __ddiv_rn(__dadd_rn(dsigma, -d0), __dadd_rn(d1, -d0));
            if (fabs(dalfa) > 1.1 || dalfa < 0.0) {
                h = 0.0;
            } else {
                const double a = __dmul_rn(ddepu[(size_t)k * pitch], dalfa);
                const double b = __dmul_rn(__dadd_rn(1.0, -dalfa), ddepu[(size_t)(k - 1) * pitch]);
                h = __dadd_rn(a, b);
            }
            break;
        }
        d0 = d1;
    }
    const double e = (double)eu;
    double w = 0.0;
    for (int k = 1; k <= nk - 1; ++k) {
        const float gw1 = ddepw ? ddepw[(size_t)k * pitch] : gdepw[k];
        const double u = (double)zu[(size_t)(k - 1) * pitch];
        if ((double)gw1 < h) {
            w = __dadd_rn(w, __dmul_rn(__dmul_rn(e, (double)de3[(size_t)(k - 1) * pitch]), u));
        } else {
            const float gw0 = ddepw ? ddepw[(size_t)(k - 1) * pitch] : gdepw[k - 1];
            w = __dadd_rn(w, __dmul_rn(__dmul_rn(e, __dadd_rn(h, -(double)gw0)), u));
            break;
        }
    }
    h_out = h;
    w_out = w;
}

// bin b of one section, by one warp (:621-627): coalesced differences (stored to dwtrpbin unless NULL), then the whole
// warp adds them in ji order (what SUM does) through shuffles; every lane returns the sum
__device__ __forceinline__ double sigtrp_bin_sum(const double *dwtrp, double *dwtrpbin, size_t pitch, int npts, int b, int lane)
{
    double s = 0.0;
    for (int i0 = 0; i0 < npts; i0 += 32) {
        const int i = i0 + lane;
        double d = 0.0;
        if (i < npts) {
            d = __dadd_rn(dwtrp[(size_t)(b + 1) * pitch + i], -dwtrp[(size_t)b * pitch + i]);
            if (dwtrpbin) dwtrpbin[(size_t)b * pitch + i] = d;
        }
        const int n = min(32, npts - i0);
        for (int l = 0; l < n; ++l) s = __dadd_rn(s, __shfl_sync(kFull, d, l));
    }
    return s;
}

// ---- one section (cdfsigtrp_gpu_section): four launches
template <int MODE>
__global__ void sigtrp_density_kernel(const SigtrpParams p)
{
    const size_t n = (size_t)p.nk * p.npts;
    for (size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (size_t)gridDim.x * blockDim.x)
        p.dsig[(size_t)p.npts + c] = sigtrp_density<MODE>(p.zt[c], p.zs[c], p.zmask[c], p.dlh, p.dlref);
}

__global__ void sigtrp_fill_kernel(const SigtrpParams p)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.npts) return;
    sigtrp_fill_column(p.dsig + i, p.zmask + i, p.npts, p.nk);
}

__global__ void sigtrp_iso_kernel(const SigtrpParams p)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x, iso = blockIdx.y;
    if (i >= p.npts) return;
    double h, w;
    sigtrp_iso_column<false>(p.ddepu + i, p.dsig + i, nullptr, p.de3 + i, p.zu + i, p.ddepw ? p.ddepw + i : nullptr, p.gdepw,
                             p.eu[i], p.lev[iso], p.npts, p.npk, p.nk, h, w);
    p.dhiso[(size_t)iso * p.npts + i] = h;
    p.dwtrp[(size_t)iso * p.npts + i] = w;
}

// one warp per bin
__global__ void sigtrp_bins_kernel(const SigtrpParams p)
{
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (b >= p.nbins) return;   // warp-uniform
    const double s = sigtrp_bin_sum(p.dwtrp, p.dwtrpbin, p.npts, p.npts, b, lane);
    if (lane == 0) p.dtrpbin[b] = s;
}

// ---- a list of sections cut from whole 3-D fields (cdfsigtrp_gpu_sections_device): four launches whatever the number of
// sections.  The columns of every section are concatenated into one axis of ncol columns (section s owns
// sec_off[s] .. sec_off[s+1]-1, in the reference's column order); every per-column array is [level][ncol].
struct SigtrpBatch {
    const float *zu3, *zv3, *zt3, *zs3;   // the caller's fields (npk, ny, nx); zu3 / zv3 read by meridional / zonal sections
    const int *col_sec;                   // (ncol) section of a column
    const int *col_ia, *col_ib;           // (ncol) j*nx+i of the two T/S points averaged; the velocity point is col_ia
    const int *sec_off, *sec_merid;       // (nsec+1) column offsets; (nsec) 1 = meridional (U, zspu, masked zt)
    int *nk;                              // (nsec) levels used, written by sigtrp_sections_nk_kernel; 0 for a skipped section
    int32_t *nk_out;                      // (nsec) the caller's copy of nk, or NULL
    const float *eu, *de3, *gdepw;        // (ncol), (npk, ncol), (npk)
    const double *ddepu, *lev;            // (npk+1, ncol), (nbins+1)
    float *zu, *zt, *zs, *zmask;          // (npk, ncol)
    double *dsig, *dwtrp;                 // (npk+1, ncol) before the land fill (row 0 unused), (nbins+1, ncol)
    double *dtrpbin;                      // (nsec, nbins): the caller's d_dtrpbin
    float zspu, zspv, zsps;
    double dlh, dlref;
    size_t nxy;
    int ncol, npk, nsec, nbins;
};

// gather + preparation (:428-460 / :521-555) + density, one thread per (level, column), every level
template <int MODE>
__global__ void sigtrp_sections_prep_kernel(const SigtrpBatch b)
{
    const size_t n = (size_t)b.npk * b.ncol;
    for (size_t cell = (size_t)blockIdx.x * blockDim.x + threadIdx.x; cell < n; cell += (size_t)gridDim.x * blockDim.x) {
        const int k = (int)(cell / b.ncol), c = (int)(cell - (size_t)k * b.ncol);
        const bool merid = b.sec_merid[b.col_sec[c]] != 0;
        const size_t lev = (size_t)k * b.nxy;
        const size_t ia = lev + b.col_ia[c], ib = lev + b.col_ib[c];
        float u = (merid ? b.zu3 : b.zv3)[ia];
        if (u == (merid ? b.zspu : b.zspv)) u = 0.0f;
        const float sa = b.zs3[ia], sb = b.zs3[ib];
        const float m = (sa == b.zsps || sb == b.zsps) ? 0.0f : 1.0f;
        const float s = __fmul_rn(__fmul_rn(0.5f, __fadd_rn(sa, sb)), m);
        float t = __fmul_rn(0.5f, __fadd_rn(b.zt3[ia], b.zt3[ib]));
        if (merid) t = __fmul_rn(t, m);   // only the meridional branch masks the mean temperature (:555)
        b.zu[cell] = u;
        b.zt[cell] = t;
        b.zs[cell] = s;
        b.zmask[cell] = m;
        b.dsig[(size_t)b.ncol + cell] = sigtrp_density<MODE>(t, s, m, b.dlh, b.dlref);
    }
}

// nk (:449-454): the first level whose REAL(4) sum of zs over the section, in column order, is 0; npk when there is none.
// One block per section, one thread per level; 0 for a skipped section.
__global__ void sigtrp_sections_nk_kernel(const SigtrpBatch b)
{
    const int s = blockIdx.x, off = b.sec_off[s], npts = b.sec_off[s + 1] - off;
    __shared__ int nk_s;
    if (threadIdx.x == 0) nk_s = b.npk;
    __syncthreads();
    for (int k = threadIdx.x; k < b.npk; k += blockDim.x) {
        const float *row = b.zs + (size_t)k * b.ncol + off;
        float sum = 0.0f;
        for (int j = 0; j < npts; ++j) sum = __fadd_rn(sum, row[j]);
        if (sum == 0.0f) atomicMin(&nk_s, k + 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const int nk = npts > 0 ? nk_s : 0;
        b.nk[s] = nk;
        if (b.nk_out) b.nk_out[s] = nk;
    }
}

// land fill, isopycnal depth and cumulative transport, one thread per (column, class limit), nk from the device table
__global__ void sigtrp_sections_iso_kernel(const SigtrpBatch b)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x, iso = blockIdx.y;
    if (c >= b.ncol) return;
    double h, w;
    sigtrp_iso_column<true>(b.ddepu + c, b.dsig + c, b.zmask + c, b.de3 + c, b.zu + c, nullptr, b.gdepw, b.eu[c], b.lev[iso], b.ncol,
                            b.npk, b.nk[b.col_sec[c]], h, w);
    b.dwtrp[(size_t)iso * b.ncol + c] = w;
}

// one warp per (section, bin): the section's columns in order, as sigtrp_bins_kernel; a skipped section's row is 0
__global__ void sigtrp_sections_bins_kernel(const SigtrpBatch b)
{
    const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (wid >= b.nsec * b.nbins) return;   // warp-uniform
    const int s = wid / b.nbins, bin = wid - s * b.nbins;
    const int off = b.sec_off[s], npts = b.sec_off[s + 1] - off;
    const double sum = sigtrp_bin_sum(b.dwtrp + off, nullptr, b.ncol, npts, bin, lane);
    if (lane == 0) b.dtrpbin[(size_t)s * b.nbins + bin] = sum;
}

}  // namespace cdfgpu
