// moc_decomp.cuh -- cdfmoc -decomp: barotropic / geostrophic-shear / ageostrophic split of the MOC.
// Replaces src/cdfmoc.f90:353,360-365,390-517 (SURVEY.md App. E.1).  Not a bandwidth showcase: six small kernels, a fixed
// number of launches whatever nz is, that reproduce the reference's REAL(4)/REAL(8) chains operation by operation; the
// zonal sums reuse K1 (noscan).
//   dvbt(i,j)   = sum_k dble(fl32(e3m*zv)) / hdep            hdep = fl32 running sum of e3m          (:363-364,:397-401)
//   dmoc_bt     = -sum_i dble(fl32(fl32(e1v*e3m)*mask)) * dvbt, scanned /1.d6                        (:403-419)
//   zsig0       = fl32(sigmai_dep(T,S,gdept(k)) * tmask), every level in one launch                  (:443)
//   dgeo, dvgeo, zv_geo : 4-point stencil, vertical recurrence from the bottom, one thread per column (:447-461)
//   dmoc_sh     = K1 on zv_geo  -  (weighted sum with the vertical mean of zv_geo), scanned /1.e6    (:464-510)
//   dmoc_ag     = dmoc - dmoc_sh - dmoc_bt                                                           (:516)
#pragma once
#include "common.cuh"
#include "eos_device.cuh"   // exact EOS chain (eos_sigma_exact)

namespace cdfgpu {

// vertical mean of fl32(e3m*zv): one thread per column; `descending` = the level order the reference sums in
__global__ void decomp_vbar_kernel(const float *__restrict__ e3m, const float *__restrict__ zv, size_t nxy, int nzm1,
                                   int descending, float *__restrict__ hdep, int write_hdep, double *__restrict__ dvbt)
{
    for (size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x; c < nxy; c += (size_t)gridDim.x * blockDim.x) {
        double dv = 0.0;
        float hd = 0.0f;
        for (int n = 0; n < nzm1; ++n) {
            const int k = descending ? nzm1 - 1 - n : n;
            const float e = e3m[(size_t)k * nxy + c];
            dv = __dadd_rn(dv, (double)__fmul_rn(e, zv[(size_t)k * nxy + c]));
            hd = __fadd_rn(hd, e);
        }
        if (write_hdep) hdep[c] = hd;
        const float h = write_hdep ? hd : hdep[c];
        dvbt[c] = (h != 0.0f) ? __ddiv_rn(dv, (double)h) : 0.0;
    }
}

// raw(b,j,k) = -sum_i dble(fl32(fl32(e1v*e3m)*real(mask_b))) * w(i,j): one warp per (j,k) row
template <int NB>
__global__ void decomp_weighted_rows_kernel(const float *__restrict__ area, const int16_t *__restrict__ ibmask,
                                            const double *__restrict__ w, int nx, int ny, int nzm1,
                                            double *__restrict__ raw)
{
    const int lane = threadIdx.x & 31;
    const int nrows = ny * nzm1;
    for (int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < nrows; r += gridDim.x * (blockDim.x >> 5)) {
        const int k = r / ny, j = r - k * ny;
        double acc[NB];
#pragma unroll
        for (int b = 0; b < NB; ++b) acc[b] = 0.0;
        for (int i = lane; i < nx; i += 32) {
            const size_t c = (size_t)j * nx + i;
            const float a = area[(size_t)k * ny * nx + c];
            const double wv = w[c];
#pragma unroll
            for (int b = 0; b < NB; ++b)
                acc[b] = __dadd_rn(acc[b], -__dmul_rn((double)__fmul_rn(a, (float)ibmask[c * NB + b]), wv));
        }
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            const double t = warp_sum(acc[b]);
            if (lane == b) raw[((size_t)k * ny + j) * NB + b] = t;
        }
    }
}

// psi(k) = psi(k+1) + (raw(k) - sub(k))/1e6 from the bottom, one thread per (j,b); level nz-1 = 0
__global__ void decomp_scan_kernel(double *__restrict__ d, const double *__restrict__ sub, int nyb, int nz)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nyb) return;
    double psi = 0.0;
    d[(size_t)(nz - 1) * nyb + t] = 0.0;
    for (int k = nz - 2; k >= 0; --k) {
        double v = d[(size_t)k * nyb + t];
        if (sub) v = __dadd_rn(v, -sub[(size_t)k * nyb + t]);
        psi = __dadd_rn(psi, __ddiv_rn(v, 1.0e6));
        d[(size_t)k * nyb + t] = psi;
    }
}

__global__ void decomp_ageo_kernel(const double *__restrict__ tot, const double *__restrict__ sh,
                                   const double *__restrict__ bt, double *__restrict__ ag, size_t n)
{
    for (size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (size_t)gridDim.x * blockDim.x)
        ag[c] = __dadd_rn(__dadd_rn(tot[c], -sh[c]), -bt[c]);
}

// zsig0 = fl32(sigmai_dep(T,S,gdept(k)) * tmask) for every level at once: blockIdx.y = level k, whose reference profile is
// dl[2k] = dlh, dl[2k+1] = dlref (eos.f90:843-845, computed on the host)
__global__ void decomp_sigma_kernel(const float *__restrict__ zt, const float *__restrict__ zs,
                                    const int16_t *__restrict__ tmask, const double *__restrict__ dl, size_t nxy,
                                    float *__restrict__ sig)
{
    const int k = blockIdx.y;
    const double dlh = dl[2 * k], dlref = dl[2 * k + 1];
    const size_t o = (size_t)k * nxy;
    for (size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x; c < nxy; c += (size_t)gridDim.x * blockDim.x)
        sig[o + c] = __double2float_rn(__dmul_rn(eos_sigma_exact<false>(zt[o + c], zs[o + c], dlh, dlref), (double)tmask[o + c]));
}

// The geostrophic recurrence (:447-461), one thread per (i,j) column walking k up from the bottom level: dvgeo stays in a
// register, e1u, zcoef and the global mask byte are read once.  Per level the operations and their order are those of the
// reference's loop body, so the result does not depend on how the columns are scheduled.  Border cells of zv_geo keep
// the last V level read (:357) at every level.
__global__ void decomp_geo_column_kernel(const float *__restrict__ sig, const int16_t *__restrict__ um,
                                         const float *__restrict__ e1u, const float *__restrict__ zcoef,
                                         const int16_t *__restrict__ ibmask, int nb, const float *__restrict__ e3m,
                                         const float *__restrict__ zv_last, float *__restrict__ zvgeo, int nx, int ny,
                                         int nzm1)
{
    const size_t nxy = (size_t)nx * ny;
    const size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nxy) return;
    const int j = (int)(c / nx), i = (int)(c - (size_t)j * nx);
    if (i == 0 || i == nx - 1 || j == 0 || j == ny - 1) {
        const float v = zv_last[c];
        for (int k = 0; k < nzm1; ++k) zvgeo[(size_t)k * nxy + c] = v;
        return;
    }
    const size_t cn = c + nx;
    const float e1a = e1u[cn - 1], e1b = e1u[cn], e1c = e1u[c - 1], e1d = e1u[c];
    const double coef = (double)zcoef[c], mask = (double)ibmask[c * nb];
    double dv = 0.0;   // dvgeo of the level below (0 under the bottom level)
    for (int k = nzm1 - 1; k >= 0; --k) {
        const size_t o = (size_t)k * nxy;
        const float *s = sig + o;
        const int16_t *u = um + o;
        const int su = u[cn - 1] + u[cn] + u[c - 1] + u[c];
        const float zmsv = __fdiv_rn(1.0f, (float)(su > 1 ? su : 1));
        const float t1 = __fdiv_rn(__fmul_rn(__fsub_rn(s[cn], s[cn - 1]), (float)u[cn - 1]), e1a);
        const float t2 = __fdiv_rn(__fmul_rn(__fsub_rn(s[cn + 1], s[cn]), (float)u[cn]), e1b);
        const float t3 = __fdiv_rn(__fmul_rn(__fsub_rn(s[c], s[c - 1]), (float)u[c - 1]), e1c);
        const float t4 = __fdiv_rn(__fmul_rn(__fsub_rn(s[c + 1], s[c]), (float)u[c]), e1d);
        const double dgeo = (double)__fadd_rn(__fadd_rn(__fadd_rn(t1, t2), t3), t4);
        double d = __dmul_rn(coef, dgeo);
        d = __dmul_rn(d, (double)zmsv);
        d = __dmul_rn(d, mask);
        d = __dmul_rn(d, (double)e3m[o + c]);
        const double up = __dadd_rn(dv, d);
        zvgeo[o + c] = __double2float_rn(__dmul_rn(0.5, __dadd_rn(up, dv)));
        dv = up;
    }
}

}  // namespace cdfgpu
