// zonal_kernels.cuh -- K4 / K5: the masked zonal integral behind the sibling command lines (SURVEY.md section 8 f3).
//   K4 zonal_rows_kernel   cdfzonalsum  (src/cdfzonalsum.f90:309-322)  and cdfzonalmean (src/cdfzonalmean.f90:312-344)
//   K5 mhst_rows_kernel    cdfmhst      (src/cdfmhst.f90:303-366): vertical integral of the heat / salt transports,
//                                       then the masked zonal sums
//   K5v mhst_vpoint_kernel cdfmhst -v/-t[-s] (src/cdfmhst.f90:313-323): T and S onto V points, times V, ahead of K5
// Both are HBM-streaming reductions like K1: coalesced loads, fp64 accumulation in registers, shuffle trees, no atomics
// (bitwise reproducible).  The products follow the reference's types and association (REAL(4) or REAL(8) chains,
// never contracted: the library is built with -fmad=false); only the order of the fp64 additions along i differs from
// the reference's sequential loop.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace cdfgpu {

__device__ __forceinline__ double warp_max(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(kFull, v, o));
    return v;
}
__device__ __forceinline__ double warp_min(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(kFull, v, o));
    return v;
}

// One warp per (level k, row j).  zmask is planar [NB][ny][nx]; out / omax / omin are [NB][nk][ny].
//   MEAN = false: dtmp = dble(fl32(fl32(zmask*zmaskvar)*zv)); sum += dl_surf*dtmp; out = sum / alpha(j)
//   MEAN = true : dtmp = ((1.d0*zmask)*zmaskvar)*zv in REAL(8); sum += dl_surf*dtmp; area += (dl_surf*zmask)*zmaskvar;
//                 out = area /= 0 ? sum/area : zspval; lmax: max / min (non-zero) of dtmp as REAL(4), zspval where area == 0
// BITS: every basin mask value is exactly 0 or 1 (checked at setup): one byte per (j,i) holds the NB mask bits; the
// product chain then has only two possible values per cell, the one of a 1 and the one of a 0 (a signed zero, or NaN
// when the data are not finite): both are formed once and selected per basin, which is what the reference computes.
// The two HBM streams (zv, zmaskvar) are read with 16-byte loads, 512 contiguous bytes per warp instruction (a 128-byte
// granularity over thousands of concurrent rows thrashes the DRAM pages: 2.2 TB/s); dl_surf and the mask bytes of the
// row come from L1 / L2 (level-fastest row order: the warps of a CTA share the latitude row).
template <int NB, bool MEAN, bool BITS>
struct ZonalAcc {
    double acc[NB], area[MEAN ? NB : 1], dmax[MEAN ? NB : 1], dmin[MEAN ? NB : 1];
    float zf;   // fast path: NaN as soon as a product of the lane was not finite
    __device__ __forceinline__ void init()
    {
        zf = 0.0f;
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            acc[b] = 0.0;
            if (MEAN) { area[b] = 0.0; dmax[b] = -INFINITY; dmin[b] = INFINITY; }
        }
    }
    // Fast form of a cell for 0 / 1 basin masks and finite data (no zonal max / min): the reference adds d*dtmp(mask = 1) or
    // d*dtmp(mask = 0) = +-0 to every basin's sum; fma(t1, m, acc) with m = 1.0 / 0.0 taken from the mask bit gives
    // acc + t1 (one rounding, t1*1 is exact) and acc + (+-0) = acc -- one integer multiply and one DFMA per basin instead
    // of a bit test, two FSELs and a DADD.  With non-finite data the mask-0 term is NaN in the reference (0*Inf) but can be
    // +-0 here and vice versa: zf turns NaN then and the warp redoes the row with cell().
    __device__ __forceinline__ void cell_fast(float v, float mv, double d, unsigned bits)
    {
        double t1, a1 = 0.0;
        if (!MEAN) {
            const float p1 = __fmul_rn(mv, v);   // fl32(fl32(1*mv)*v)
            zf = __fmaf_rn(p1, 0.0f, zf);
            t1 = __dmul_rn(d, (double)p1);
        } else {
            zf = __fmaf_rn(mv, 0.0f, __fmaf_rn(v, 0.0f, zf));
            const double dmv = (double)mv;
            t1 = __dmul_rn(d, __dmul_rn(dmv, (double)v));
            a1 = __dmul_rn(d, dmv);
        }
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            const double m = __hiloint2double((int)((bits & (1u << b)) * (0x3FF00000u >> b)), 0);   // 1.0 or 0.0
            acc[b] = __fma_rn(t1, m, acc[b]);
            if (MEAN) area[b] = __fma_rn(a1, m, area[b]);
        }
    }
    // one cell: v = zv, mv = zmaskvar, d = dl_surf, bits = packed masks (BITS) or pz = the cell in plane 0 (!BITS)
    __device__ __forceinline__ void cell(float v, float mv, double d, unsigned bits, const float *pz, size_t nxy, int lmax)
    {
        if (BITS) {
            if (!MEAN) {
                const double t1 = __dmul_rn(d, (double)__fmul_rn(__fmul_rn(1.0f, mv), v));
                const double t0 = __dmul_rn(d, (double)__fmul_rn(__fmul_rn(0.0f, mv), v));
#pragma unroll
                for (int b = 0; b < NB; ++b) acc[b] = __dadd_rn(acc[b], ((bits >> b) & 1u) ? t1 : t0);
            } else {
                const double dmv = (double)mv, dv = (double)v;
                const double x1 = __dmul_rn(__dmul_rn(1.0, dmv), dv), x0 = __dmul_rn(__dmul_rn(0.0, dmv), dv);
                const double t1 = __dmul_rn(d, x1), t0 = __dmul_rn(d, x0);
                const double a1 = __dmul_rn(__dmul_rn(d, 1.0), dmv), a0 = __dmul_rn(__dmul_rn(d, 0.0), dmv);
#pragma unroll
                for (int b = 0; b < NB; ++b) {
                    const bool on = ((bits >> b) & 1u) != 0u;
                    const double dtmp = on ? x1 : x0;
                    acc[b] = __dadd_rn(acc[b], on ? t1 : t0);
                    area[b] = __dadd_rn(area[b], on ? a1 : a0);
                    if (lmax) {   // NaN never wins a Fortran MAX/MIN started from a number: fmax / fmin behave the same
                        dmax[b] = fmax(dmax[b], dtmp);
                        if (dtmp != 0.0) dmin[b] = fmin(dmin[b], dtmp);
                    }
                }
            }
        } else {
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                const float m = __ldg(pz + (size_t)b * nxy);
                if (!MEAN) {
                    const float p = __fmul_rn(__fmul_rn(m, mv), v);
                    acc[b] = __dadd_rn(acc[b], __dmul_rn(d, (double)p));
                } else {
                    const double dm = (double)m;
                    const double dtmp = __dmul_rn(__dmul_rn(dm, (double)mv), (double)v);
                    acc[b] = __dadd_rn(acc[b], __dmul_rn(d, dtmp));
                    area[b] = __dadd_rn(area[b], __dmul_rn(__dmul_rn(d, dm), (double)mv));
                    if (lmax) {
                        dmax[b] = fmax(dmax[b], dtmp);
                        if (dtmp != 0.0) dmin[b] = fmin(dmin[b], dtmp);
                    }
                }
            }
        }
    }
};

template <int NB, bool MEAN, bool BITS>
__global__ void __launch_bounds__(256) zonal_rows_kernel(const float *__restrict__ zv, const float *__restrict__ mvar,
                                                         const float *__restrict__ zmask, const uint8_t *__restrict__ zbits,
                                                         const double *__restrict__ dl, const float *__restrict__ alpha, int nx,
                                                         int ny, int nk, float zspval, int lmax, double *__restrict__ out,
                                                         float *__restrict__ omax, float *__restrict__ omin)
{
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    const size_t nrows = (size_t)nk * ny;
    const size_t nxy = (size_t)nx * ny;
    const uint64_t pol = make_evict_first_policy();
    for (size_t r = (size_t)blockIdx.x * wpb + (threadIdx.x >> 5); r < nrows; r += (size_t)gridDim.x * wpb) {
        // level fastest: the warps of a CTA work on the same latitude row
        const int j = (int)(r / nk), k = (int)(r - (size_t)j * nk);
        const size_t e0 = ((size_t)k * ny + j) * nx;
        const float *pv = zv + e0, *pm = mvar + e0;
        const double *pd = dl + (size_t)j * nx;
        const float *pz = zmask + (size_t)j * nx;
        const uint8_t *pb = zbits + (size_t)j * nx;
        ZonalAcc<NB, MEAN, BITS> A;
        const int head = min((int)((4 - (e0 & 3)) & 3), nx);   // scalar cells in front of the first 16-byte boundary
        const int nvec = (nx - head) >> 2;
        const int tail0 = head + 4 * nvec;
        auto sweep = [&](auto fast_tag) {
            constexpr bool FAST = decltype(fast_tag)::value;
            A.init();
            {   // head and tail cells (at most 3 + 3), one per lane
                int i = -1;
                if (lane < head) i = lane;
                else if (lane - head < nx - tail0) i = tail0 + lane - head;
                if (i >= 0) {
                    if (FAST) A.cell_fast(__ldg(pv + i), __ldg(pm + i), __ldg(pd + i), (unsigned)__ldg(pb + i));
                    else A.cell(__ldg(pv + i), __ldg(pm + i), __ldg(pd + i), BITS ? (unsigned)__ldg(pb + i) : 0u, pz + i, nxy, lmax);
                }
            }
#pragma unroll 2
            for (int vi = lane; vi < nvec; vi += 32) {
                const int i = head + 4 * vi;
                const float4 v = ld_stream_f4(reinterpret_cast<const float4 *>(pv + i), pol);
                const float4 m = __ldg(reinterpret_cast<const float4 *>(pm + i));
                const float vv[4] = {v.x, v.y, v.z, v.w}, mm[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    if (FAST) A.cell_fast(vv[c], mm[c], __ldg(pd + i + c), (unsigned)__ldg(pb + i + c));
                    else A.cell(vv[c], mm[c], __ldg(pd + i + c), BITS ? (unsigned)__ldg(pb + i + c) : 0u, pz + i + c, nxy, lmax);
                }
            }
        };
        bool fast = BITS && !lmax;   // warp-uniform
        if (fast) {
            sweep(std::true_type{});
            if (__any_sync(kFull, A.zf != A.zf)) fast = false;   // a non-finite product somewhere in the row: the literal chain
        }
        if (!fast) sweep(std::false_type{});
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            const double s = warp_sum(A.acc[b]);
            const size_t o = ((size_t)b * nk + k) * ny + j;
            if (!MEAN) {
                if (lane == 0) out[o] = s / (double)(alpha ? alpha[j] : 1.0f);
            } else {
                const double a = warp_sum(A.area[b]);
                if (lane == 0) out[o] = (a != 0.0) ? s / a : (double)zspval;
                if (lmax) {
                    const double mx = warp_max(A.dmax[b]), mn = warp_min(A.dmin[b]);
                    if (lane == 0) {   // rzomax starts at -1.e20, rzomin at 1.e20 (REAL(4)); REAL(4) <- REAL(8) rounding is monotone
                        omax[o] = (a == 0.0) ? zspval : (float)fmax((double)(-1.e20f), mx);
                        omin[o] = (a == 0.0) ? zspval : (float)fmin((double)(1.e20f), mn);
                    }
                }
            }
        }
    }
}

// setup: dl_surf = (1.d0*e1)*e2 (cdfzonalsum.f90:257) and the basin planes (nb,nx,ny) basin-fastest -> planar [nb][ny][nx]
__global__ void zonal_prep_kernel(const float *__restrict__ e1, const float *__restrict__ e2, const float *__restrict__ zmask_in,
                                  int nb, size_t nxy, double *__restrict__ dl, float *__restrict__ zmask_planar)
{
    for (size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x; c < nxy; c += (size_t)gridDim.x * blockDim.x) {
        dl[c] = __dmul_rn(__dmul_rn(1.0, (double)e1[c]), (double)e2[c]);
        for (int b = 0; b < nb; ++b) zmask_planar[(size_t)b * nxy + c] = zmask_in[c * nb + b];
    }
}

// K5v: the V-point products of cdfmhst's separate-file mode, per cell of (nz,ny,nx) records zv, zt, zs:
//   zvt = fl32(fl32(0.5*fl32(zt(j)+zt(j+1)))*zv), zvs likewise; the last row (npjglo) stays 0 (cdfmhst.f90:313-323).
// Each operation rounds on its own (__fadd_rn / __fmul_rn: no FFMA), in the host loop's order.  A CTA walks whole (k,j)
// rows so that no cell needs a division; the row j+1 of zt / zs is the next row's load, served from L2 on the way.
// HBM-bound: 12 B read and 8 B written per cell.
__global__ void __launch_bounds__(256) mhst_vpoint_kernel(const float *__restrict__ zv, const float *__restrict__ zt,
                                                          const float *__restrict__ zs, int nx, int ny, int nz,
                                                          float *__restrict__ vt, float *__restrict__ vs)
{
    const size_t rows = (size_t)nz * ny;
    for (size_t r = blockIdx.x; r < rows; r += gridDim.x) {
        const bool last = (int)(r % (size_t)ny) == ny - 1;
        const size_t c0 = r * (size_t)nx;
        for (int i = threadIdx.x; i < nx; i += blockDim.x) {
            const size_t c = c0 + i;
            if (last) { vt[c] = 0.f; vs[c] = 0.f; continue; }
            const float v = __ldcs(zv + c);
            const float th = __fmul_rn(0.5f, __fadd_rn(zt[c], zt[c + nx]));
            const float sh = __fmul_rn(0.5f, __fadd_rn(zs[c], zs[c + nx]));
            __stcs(vt + c, __fmul_rn(th, v));
            __stcs(vs + c, __fmul_rn(sh, v));
        }
    }
}

// K5: one CTA per latitude row j; a thread owns up to MAXC columns (i = tid + c*blockDim) and integrates them over the
// levels in the reference's order:  dtrph += (dble(fl32(fl32(zvt*e1v)*e3v))*1000.)*4000. ; dtrps += dble(fl32(fl32(zvs*e1v)*e3v))
// After the last level (every level with zdim) the masked zonal sums: global over i = 2..nx-1 with vmask(k=1), the basins
// over all i.  masks: planar [4][ny][nx] (glo, atl, pac, ind; planes of absent basins are zero).  heat, salt: [nlev][4][ny].
// The three HBM streams of a level (zvt, zvs, e3v rows) are staged in shared memory with 16-byte cp.async copies, double
// buffered: the next level is in flight while this one is integrated, and every warp instruction moves 512 contiguous
// bytes whatever the alignment of the row (the misalignment (k*nx*ny + j*nx) mod 4 changes from level to level, so a
// thread cannot keep fixed columns AND aligned vector loads without the staging).
template <int MAXC>
__global__ void __launch_bounds__(1024) mhst_rows_kernel(const float *__restrict__ zvt, const float *__restrict__ zvs,
                                                         const float *__restrict__ e1v, const float *__restrict__ e3v,
                                                         const float *__restrict__ masks, int nx, int ny, int nz, int zdim,
                                                         int nmask, int pitch, double *__restrict__ heat, double *__restrict__ salt)
{
    extern __shared__ float s_stage[];   // [2 buffers][3 arrays][pitch]
    __shared__ double s_red[32][8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5, nthreads = blockDim.x;
    const size_t nxy = (size_t)nx * ny;
    for (int j = blockIdx.x; j < ny; j += gridDim.x) {
        auto issue = [&](int k, int buf) {
            const size_t base = (size_t)k * nxy + (size_t)j * nx;
            const int sh = (int)(base & 3);
            const int head = min((4 - sh) & 3, nx), nvec = (nx - head) >> 2, tail0 = head + 4 * nvec;
            const float *src[3] = {zvt + base, zvs + base, e3v + base};
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                float *dst = s_stage + (size_t)(buf * 3 + a) * pitch + sh;   // element i lives at dst[i]: dst + head is 16-byte aligned
                for (int vi = tid; vi < nvec; vi += nthreads) cp_async16(dst + head + 4 * vi, src[a] + head + 4 * vi);
                if (tid < head) cp_async4(dst + tid, src[a] + tid);
                else if (tid - head < nx - tail0) cp_async4(dst + tail0 + tid - head, src[a] + tail0 + tid - head);
            }
            cp_async_commit();
        };
        double th[MAXC], ts[MAXC];
        float e1[MAXC];
#pragma unroll
        for (int c = 0; c < MAXC; ++c) {
            const int i = tid + c * nthreads;
            th[c] = 0.0; ts[c] = 0.0;
            e1[c] = (i < nx) ? __ldg(e1v + (size_t)j * nx + i) : 0.0f;
        }
        issue(0, 0);
        for (int k = 0; k < nz; ++k) {
            if (k + 1 < nz) {
                issue(k + 1, (k + 1) & 1);
                cp_async_wait<1>();
            } else {
                cp_async_wait<0>();
            }
            __syncthreads();
            const int sh = (int)(((size_t)k * nxy + (size_t)j * nx) & 3);
            const float *bvt = s_stage + (size_t)((k & 1) * 3 + 0) * pitch + sh, *bvs = bvt + pitch, *be3 = bvs + pitch;
#pragma unroll
            for (int c = 0; c < MAXC; ++c) {
                const int i = tid + c * nthreads;
                if (i < nx) {
                    const float e3 = be3[i];
                    const float h = __fmul_rn(__fmul_rn(bvt[i], e1[c]), e3);
                    const float s = __fmul_rn(__fmul_rn(bvs[i], e1[c]), e3);
                    th[c] = __dadd_rn(th[c], __dmul_rn(__dmul_rn((double)h, 1000.0), 4000.0));
                    ts[c] = __dadd_rn(ts[c], (double)s);
                }
            }
            if (zdim || k == nz - 1) {
                double part[8];
#pragma unroll
                for (int m = 0; m < 4; ++m) {
                    double sh_ = 0.0, ss = 0.0;
                    if (m < nmask) {
#pragma unroll
                        for (int c = 0; c < MAXC; ++c) {
                            const int i = tid + c * nthreads;
                            const bool in = (m == 0) ? (i >= 1 && i < nx - 1) : (i < nx);
                            if (in) {
                                const double mk = (double)__ldg(masks + (size_t)m * nxy + (size_t)j * nx + i);
                                sh_ = __dadd_rn(sh_, __dmul_rn(th[c], mk));
                                ss = __dadd_rn(ss, __dmul_rn(ts[c], mk));
                            }
                        }
                    }
                    part[2 * m] = warp_sum(sh_);
                    part[2 * m + 1] = warp_sum(ss);
                }
                if (lane == 0) {
#pragma unroll
                    for (int q = 0; q < 8; ++q) s_red[warp][q] = part[q];
                }
                __syncthreads();
                if (tid < 8) {
                    double t = 0.0;
                    for (int w = 0; w < nwarps; ++w) t += s_red[w][tid];   // fixed order: deterministic
                    const int lev = zdim ? k : 0, m = tid >> 1;
                    double *dst = (tid & 1) ? salt : heat;
                    dst[((size_t)lev * 4 + m) * ny + j] = t;
                }
            }
            __syncthreads();   // this level's buffer (and s_red) may be overwritten from the next trip on
        }
    }
}

}  // namespace cdfgpu
