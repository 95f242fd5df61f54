// moc_kernel.cuh -- K1: depth-space MOC.  Replaces the loop nest src/cdfmoc.f90:352-388.
//
//   T(b,j,k) = sum_i -dble( fl32( fl32( fl32(e1v*e3m) * real(ibmask(b)) ) * zv ) )       (cdfmoc.f90:373-374)
//   psi(b,j,nz) = 0 ; psi(b,j,k) = psi(b,j,k+1) + T(b,j,k)/1.d6 , k = nz-1..1            (cdfmoc.f90:385)
//
// Design (HBM-bound streaming reduction, 8 algorithmic bytes per level-cell):
//   * `area` = fl32(e1v*e3m) is precomputed once at setup and stays resident; the basin masks are packed into one byte
//     per (j,i) (bit b = basin b) and kept L2-resident, so a record costs 4 B (V) + 4 B (area) per cell.
//   * One warp owns one (j,k) row at a time; work units (`chunk` consecutive levels of one latitude row, j-major) are
//     handed out dynamically through 32 sharded ticket counters with stealing (a same-address L2 atomic completes only
//     every ~3.6 ns) to a persistent grid of 3 CTAs per SM; the next ticket is requested one unit ahead.
//   * Loads are 16-byte streaming loads on the FLAT array (rows of the ORCA grids are only 8-byte aligned, so vectors may
//     straddle row ends): the mask words are stored in 4 pre-shifted planes, one word per vector, aligned with the float4
//     lanes.  A word holds the vector's lead basin byte and which of its in-row cells carry it ("kept").
//   * Per vector: 4 FMUL (fl32 products, exactly the reference's chain when the mask is 0/1; cells not kept enter with
//     area 0), their fp64 sum, and per basin ONE DFMA whose multiplier (-1.0 / -0.0) is built from the lead byte.  The few
//     in-row cells with another non-zero byte are listed per row, one per lane, and added cell by cell.  fp64 lane
//     partials -> warp shuffle tree.
//   * Exactness guard: the fast path equals the reference chain whenever masks are in {0,1} and the products are
//     finite.  A NaN/Inf anywhere in the row is detected for free (fma(p,0,flag)) and the warp then redoes the
//     row with the literal multiply chain (row_general_store), which is also the path for non-binary masks.
//   * The raw sums go to the output slab; the warp that completes the last level of a column j performs the
//     bottom-up recurrence in the reference's sequential order (lanes = basins) -- no second kernel.
//   * Consecutive launches of a stream overlap (programmatic dependent launch): see the kernel body.
#pragma once
#include "common.cuh"

namespace cdfgpu {

struct MocParams {
    const float *__restrict__ zv;       // (nz-1, ny, nx) one time record, levels 1..nz-1
    const float *__restrict__ area;     // (nz-1, ny, nx) fl32(e1v*e3m)
    const uint32_t *__restrict__ nzvec; // bit q&31 of word q>>5: the flat area vector q (floats 4q..4q+3) has a non-zero word
    const uint32_t *__restrict__ maskw; // [4][ny][pitchw] per vector: basin bytes and their cells (pack_masks), copy s shifted by s cells
    const uint32_t *__restrict__ exs;   // [4][ny][32] exceptions of each row (pack_masks): (i << 8) | basin byte, 0 = none
    const int16_t *__restrict__ ibmask; // (ny, nx, nb) for the general path
    double *__restrict__ out;           // (nz, ny, nb)
    int *tickets;                       // [2][kTicketShards*kTicketStride] unit tickets (ping-pong between launches)
    int *col_done;                      // [ny] rows finished per column j (self-resetting)
    int nx, ny, nz, pitchw;
    int parity;                         // launch generation mod 3 selecting tickets[parity]; this launch re-arms (parity+1)%3
    int pdl;                            // launched with programmatic stream serialization: may overlap the previous launch's tail
    int pdl_early;                      // ... and the inputs were complete before the predecessor was launched: loads may precede the wait
    int nrec;                           // records of this launch (1, or a batch: cdfmoc_gpu_compute_device_batch)
    const float *const *zv_list;        // batch: [nrec] records (device array of device pointers); null for a single record
    double *const *out_list;            // batch: [nrec] result slabs; col_done then holds nrec*ny counters
    int chunk;                          // consecutive levels of one column handed out per ticket
    int jsplit;                         // columns j >= jsplit are handed out ONE level per ticket (short tail), see kernel
    int general;                        // 1: masks are not 0/1 (or area not finite) -> literal chain everywhere
    int noscan;                         // 1: leave the raw zonal sums in `out` (-decomp combines before integrating)
};

constexpr int kMocThreads = 256;
constexpr int kTicketShards = 32;   // sharded work counters (see moc_zonal_scan_kernel)
constexpr int kTicketStride = 32;   // ints between shards: one 128-byte line each

// acc[b] -= d for every basin b whose bit is set in `bits`.  Written as ONE fused multiply-add per basin with a
// multiplier of -1.0 or -0.0 built from the bit (only the high word differs): fma(d,-1,acc) == acc - d and
// fma(d,-0,acc) == acc, both exactly.  The plain C++ conditional (and a predicated PTX sub) is lowered by ptxas to an
// unconditional DADD plus two FSELs per basin, which made FSEL 37% of all issued instructions (profiles/r01_k1v1_opmix.txt).
template <int NB>
__device__ __forceinline__ void sub_by_bits(double (&acc)[NB], double d, uint32_t bits)
{
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const int hi = (bits & (1u << b)) ? (int)0xBFF00000 : (int)0x80000000;
        acc[b] = fma(d, __hiloint2double(hi, 0), acc[b]);
    }
}

// One flat 16-byte vector: mword = lead byte M | kept cells << 8 (pack_masks).  A cell that is not kept (byte 0, outside
// the row, or an exception) enters with area 0: its product is +-0, or NaN exactly when its V is NaN / Inf -- what the
// reference's fl32(fl32(area*0)*v) gives for a byte-0 cell; the flag then sends the row to the literal chain.  The kept
// products are summed in fp64 in a fixed order and pushed into the basins of M once.
template <int NB>
__device__ __forceinline__ void moc_vector(float4 a, float4 v, uint32_t mword, double (&acc)[NB], float &badf)
{
    const float p0 = __fmul_rn((mword & 0x100u) ? a.x : 0.0f, v.x);
    const float p1 = __fmul_rn((mword & 0x200u) ? a.y : 0.0f, v.y);
    const float p2 = __fmul_rn((mword & 0x400u) ? a.z : 0.0f, v.z);
    const float p3 = __fmul_rn((mword & 0x800u) ? a.w : 0.0f, v.w);
    badf = __fmaf_rn(p0, 0.0f, badf);  // NaN iff a product is NaN/Inf, else unchanged
    badf = __fmaf_rn(p1, 0.0f, badf);
    badf = __fmaf_rn(p2, 0.0f, badf);
    badf = __fmaf_rn(p3, 0.0f, badf);
    sub_by_bits<NB>(acc, (((double)p0 + (double)p1) + (double)p2) + (double)p3, mword);
}

// Fast path: exact for 0/1 masks and finite products, up to the order of the fp64 sums.  Returns lane partial sums.
template <int NB, int kMocUnroll>
__device__ __forceinline__ void row_sums_fast(const MocParams &p, const float *__restrict__ zv, int j, int k, int lane, uint64_t pol,
                                              double (&acc)[NB], float &badf)
{
    const size_t e0 = ((size_t)k * p.ny + j) * (size_t)p.nx;
    const int s = (int)(e0 & 3);
    const size_t a0 = e0 - s;
    const int nvec = (s + p.nx + 3) >> 2;
    const unsigned q0 = (unsigned)(a0 >> 2);   // flat vector index of the row's first vector (< 2^32: checked at setup)
    const unsigned m0 = (unsigned)(s * p.ny + j) * (unsigned)p.pitchw;
    // the row's first 32 exceptions, one per lane: the entry read now, its area and V with the first vectors, its product
    // added after them (a load chain at the row's end would stall the warp there)
    const uint32_t xs = __ldg(p.exs + (((size_t)s * p.ny + j) << 5) + lane);
    float xa = 0.0f, xv = 0.0f;
    if (xs == ~0u) badf = __int_as_float(0x7fc00000);   // more than 32 exceptions: the row takes the literal chain

    for (int b0 = 0; b0 < nvec; b0 += kWarp * kMocUnroll) {   // warp-uniform trip count: the vote below needs every lane
        const int v0 = b0 + lane;
        float4 vv[kMocUnroll], aa[kMocUnroll];
        uint32_t mm[kMocUnroll];
        const unsigned q = q0 + v0;
        const float4 *__restrict__ v4 = reinterpret_cast<const float4 *>(zv) + q;
        const float4 *__restrict__ a4 = reinterpret_cast<const float4 *>(p.area) + q;
        const uint32_t *__restrict__ mw = p.maskw + (m0 + v0);
        // Zero-area vectors: vector q + 32u has bit q & 31 of word (q >> 5) + u.
        const uint32_t *__restrict__ nzw = p.nzvec + (q >> 5);
        unsigned nzb = 0u;
#pragma unroll
        for (int u = 0; u < kMocUnroll; ++u)
            if (v0 + u * kWarp < nvec && (__ldg(nzw + u) >> (q & 31) & 1u)) nzb |= 1u << u;
#pragma unroll
        for (int u = 0; u < kMocUnroll; ++u) {
            if (v0 + u * kWarp < nvec) {
                vv[u] = ld_stream_f4(v4 + u * kWarp, pol);
                mm[u] = __ldg(mw + u * kWarp);
            } else {
                vv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                mm[u] = 0u;
            }
            // an area vector whose four words are all +0.0f is not read: the zeros put in its place are the same bits.
            // (V is still read there: a NaN / Inf times a zero area poisons the row, as in the reference.)
            if (nzb & (1u << u))
                aa[u] = ld_stream_f4(a4 + u * kWarp, pol);
            else
                aa[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (b0 == 0 && xs + 1u > 1u) {
            const size_t c = e0 + (xs >> 8);
            xa = __ldg(p.area + c);
            xv = __ldg(zv + c);
        }
#pragma unroll
        for (int u = 0; u < kMocUnroll; ++u) {
            if (__any_sync(kFull, nzb & (1u << u))) {
                moc_vector<NB>(aa[u], vv[u], mm[u], acc, badf);
            } else {   // the whole warp's area is +0 here: the products only add +-0 to sums that are never -0, and
                       // v * 0 is NaN exactly when the zero-area product is
                badf = __fmaf_rn(vv[u].x, 0.0f, badf);
                badf = __fmaf_rn(vv[u].y, 0.0f, badf);
                badf = __fmaf_rn(vv[u].z, 0.0f, badf);
                badf = __fmaf_rn(vv[u].w, 0.0f, badf);
            }
        }
    }
    // The in-row cells whose byte is neither 0 nor their vector's lead byte (pack_masks; 3.7 per row of an ORCA025
    // record, at most 11), lane t taking the t-th, with the per-cell chain and the cell's own byte.  With the kept cells
    // this counts every in-row cell with a non-zero byte exactly once; the lane of an exception is fixed by its place in
    // the row's list, not by the plan.
    if (xs + 1u > 1u) {   // neither 0 (none) nor ~0 (overflow)
        const float pr = __fmul_rn(xa, xv);
        badf = __fmaf_rn(pr, 0.0f, badf);
        sub_by_bits<NB>(acc, (double)pr, xs & 0xffu);
    }
}

// General path: the literal chain of cdfmoc.f90:373-374 with INTEGER(2) mask values (any value, NaN/Inf safe).
// Handles the whole row (sums, warp reduction, store of the raw sums) so that the fast path keeps its
// accumulators in registers.
template <int NB, bool BATCH>
__device__ __noinline__ void row_general_store(const MocParams &p, int rec, int j, int k, int lane)
{
    const float *__restrict__ zv = BATCH ? p.zv_list[rec] : p.zv;
    double *__restrict__ out = BATCH ? p.out_list[rec] : p.out;
    const size_t e0 = ((size_t)k * p.ny + j) * (size_t)p.nx;
    double acc[NB];
#pragma unroll
    for (int b = 0; b < NB; ++b) acc[b] = 0.0;
    for (int i = lane; i < p.nx; i += kWarp) {
        const float a = p.area[e0 + i];
        const float v = zv[e0 + i];
        const int16_t *m = p.ibmask + ((size_t)j * p.nx + i) * NB;
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            const float t = __fmul_rn(__fmul_rn(a, (float)m[b]), v);
            acc[b] -= (double)t;
        }
    }
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const double t = warp_sum(acc[b]);
        if (lane == b) out[((size_t)k * p.ny + j) * NB + b] = t;
    }
}

// BATCH: the launch runs over several records (MocParams::nrec, zv_list, out_list); a compile-time switch, because the
// single-record kernel sits at its register budget (80 of 85 for 3 CTAs per SM) and takes p.zv / p.out / p.col_done
// straight from the constant bank.
template <int NB, int UNROLL, int MINB, bool BATCH>
__global__ void __launch_bounds__(kMocThreads, MINB) moc_zonal_scan_kernel(const MocParams p)
{
    extern __shared__ double s_scan[];  // [warps][(nz-1)*NB]
    const int lane = lane_id();
    const int warp = threadIdx.x >> 5;
    const int nzm1 = p.nz - 1;
    const uint64_t pol = make_evict_first_policy();
    // Work units = `chunk` consecutive levels of one latitude row j, numbered j-major.  They are handed out
    // dynamically, but NOT by one counter: a same-address L2 atomic completes only every ~3.6 ns on B200, so one
    // ticket per row would cost 0.27 ms per ORCA025 record by itself (measured: chunk=1 0.274 ms vs 0.160 ms).  The
    // ticket is therefore sharded over kTicketShards counters in different 128-byte lines; shard c owns the units
    // u = t*kTicketShards + c.  A warp starts on shard (global warp id mod shards) and moves on to the next shard when
    // its own runs dry (work stealing), so all shards drain together and the tail is at most one unit per warp.
    // Guided hand-out: the columns below jsplit go `chunk` levels at a time (few tickets), the last ones a single level at
    // a time, so that the tail of the launch -- warps idling while the last units finish -- is one row long, not `chunk`.
    const int chunks_per_col = (nzm1 + p.chunk - 1) / p.chunk;
    const int jsplit = min(max(p.jsplit, 0), p.ny);
    const int nbig = jsplit * chunks_per_col;
    const int nunits_rec = nbig + (p.ny - jsplit) * nzm1;   // units of one record
    const int nunits = BATCH ? nunits_rec * p.nrec : nunits_rec;   // a batch launch runs over (record, unit)
    int *tickets = p.tickets + p.parity * (kTicketShards * kTicketStride);
    {   // re-arm the next launch's counters (three sets in rotation: with programmatic dependent launch the next launch
        // starts while this one drains, and IT re-arms the set after its own -- never the one still in use here)
        int *other = p.tickets + ((p.parity + 1) % 3) * (kTicketShards * kTicketStride);
        // When the record (or the area field) may have been written by the predecessor itself -- byte swap, -vvl area build,
        // -decomp stencil, a caller's kernel right in front -- the host clears pdl_early and every CTA waits before its
        // first load: only stores are guaranteed invisible until griddepcontrol.wait, loads are not.
        if (p.pdl && (blockIdx.x == 0 || !p.pdl_early)) asm volatile("griddepcontrol.wait;" ::: "memory");
        if (blockIdx.x == 0) {
            // under PDL the set to re-arm may still be in use two launches back if CTAs of the launch in between retired
            // without work: block 0 re-arms (and only then releases the next launch) once its predecessor is complete
            if (threadIdx.x < kTicketShards) {
                other[threadIdx.x * kTicketStride] = 0;
                __threadfence();
            }
            __syncthreads();   // every warp of block 0 releases the dependents only after the re-armed counters are visible
        }
    }
    // Programmatic dependent launch: the per-launch fixed cost of this kernel (launch gap, ramp-up, and a tail in which
    // warps idle while the last units finish) is ~28 us whatever the grid -- 18 % of an ORCA025 record (tools/
    // k1_fixed_cost.py: t = 28 us + bytes / 6.7 TB/s).  Every CTA releases the next launch of the stream right away, so
    // that its CTAs fill the SMs as ours retire.  The dependent launch may take tickets, stream its first unit and reduce
    // it, but it parks the sums in shared memory and executes griddepcontrol.wait (= the previous launch has completed and
    // its writes are visible) before its first global store -- output slabs and column counters may be shared between
    // consecutive launches.
    const bool pdl = p.pdl != 0;
    if (pdl) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    bool parked = pdl && p.pdl_early && blockIdx.x != 0;   // this warp's first unit goes to the stash (the others have waited)
    double *stash = s_scan + (size_t)warp * nzm1 * NB;
    int shard = (blockIdx.x * (kMocThreads / 32) + warp) % kTicketShards;
    auto take = [&](int sh) {   // lane 0: unit index from shard sh (may be >= nunits when the shard is dry)
        return atomicAdd(tickets + sh * kTicketStride, 1) * kTicketShards + sh;
    };
    int u = 0;
    if (lane == 0) u = take(shard);
    u = __shfl_sync(kFull, u, 0);
    for (;;) {
        if (u >= nunits) {
            // this shard is exhausted: look at all shards at once (lane = shard, one L2 read) and steal from the next
            // one that still has units; when none has, the warp is done.  Counters only grow, so a stale value can
            // only cause one wasted ticket.
            const int seen = __ldcg(tickets + lane * kTicketStride) * kTicketShards + lane;
            unsigned live = __ballot_sync(kFull, seen < nunits);
            if (live == 0u) {
                // no CTA of a dependent launch retires before its predecessor is complete: the launch after this one can
                // then never run beside the one before it (the grid fills the device), whatever the amount of work
                if (pdl) asm volatile("griddepcontrol.wait;" ::: "memory");
                break;
            }
            live = (live >> shard) | (shard ? (live << (32 - shard)) : 0u);   // rotate so that bit 0 = current shard
            shard = (shard + __ffs(live) - 1) % kTicketShards;
            if (lane == 0) u = take(shard);
            u = __shfl_sync(kFull, u, 0);
            continue;
        }
        int unext = 0;
        if (lane == 0) unext = take(shard);  // request the next unit now; its latency hides behind the rows below
        int j, k0, k1;
        const float *__restrict__ zv = p.zv;
        double *__restrict__ out = p.out;
        int *col_done = p.col_done;
        int ur = u, rec = 0;
        if (BATCH) {   // the record of this unit
            rec = u / nunits_rec;
            ur = u - rec * nunits_rec;
            zv = p.zv_list[rec];   // (the slab pointer is re-read where it is used: it would not stay in a register)
            col_done += (size_t)rec * p.ny;
        }
        if (ur < nbig) {
            j = ur / chunks_per_col;
            k0 = (ur - j * chunks_per_col) * p.chunk;
            k1 = min(k0 + p.chunk, nzm1);
        } else {
            const int u2 = ur - nbig;
            const int dj = u2 / nzm1;
            j = jsplit + dj;
            k0 = u2 - dj * nzm1;
            k1 = k0 + 1;
        }
        for (int k = k0; k < k1; ++k) {
            double acc[NB];
#pragma unroll
            for (int b = 0; b < NB; ++b) acc[b] = 0.0;
            bool bad = p.general != 0;
            if (!bad) {
                float badf = 0.0f;
                row_sums_fast<NB, UNROLL>(p, zv, j, k, lane, pol, acc, badf);
                bad = __any_sync(kFull, badf != badf);
            }
            if (bad) {
                if (parked) {   // rare: flush what is parked, then the literal chain stores directly
                    if (BATCH) out = p.out_list[rec];
                    asm volatile("griddepcontrol.wait;" ::: "memory");
                    __syncwarp();
                    for (int kk = k0; kk < k; ++kk)
                        if (lane < NB) out[((size_t)kk * p.ny + j) * NB + lane] = stash[(kk - k0) * NB + lane];
                    parked = false;
                }
                row_general_store<NB, BATCH>(p, rec, j, k, lane);
            } else {
                if (BATCH) out = p.out_list[rec];
#pragma unroll
                for (int b = 0; b < NB; ++b) {
                    const double t = warp_sum(acc[b]);
                    if (lane == b) {
                        if (parked) stash[(k - k0) * NB + b] = t;
                        else out[((size_t)k * p.ny + j) * NB + b] = t;
                    }
                }
            }
        }
        if (BATCH) out = p.out_list[rec];
        if (parked) {   // first unit of this warp under PDL: the previous launch must be complete before we store
            asm volatile("griddepcontrol.wait;" ::: "memory");
            __syncwarp();
            for (int kk = k0; kk < k1; ++kk)
                if (lane < NB) out[((size_t)kk * p.ny + j) * NB + lane] = stash[(kk - k0) * NB + lane];
            parked = false;
        }
        // publish the rows, then count them; the warp that completes column j integrates it vertically.
        // Release on the counting atomic (orders this warp's row stores, made visible to lane 0 by __syncwarp) and
        // an acquire fence only in the one warp that finishes the column.
        __syncwarp();
        int done = 0;
        if (lane == 0) {
            int old;
            asm volatile("atom.add.release.gpu.global.s32 %0, [%1], %2;"
                         : "=r"(old) : "l"(col_done + j), "r"(k1 - k0) : "memory");
            done = old + (k1 - k0);
        }
        done = __shfl_sync(kFull, done, 0);
        if (done == nzm1 && p.noscan) {
            if (lane == 0) col_done[j] = 0;
        } else if (done == nzm1) {
            asm volatile("fence.acq_rel.gpu;" ::: "memory");
            double *sc = s_scan + (size_t)warp * nzm1 * NB;
            for (int t = lane; t < nzm1 * NB; t += kWarp) {
                const int kk = t / NB, b = t - kk * NB;
                sc[t] = __ldcg(out + ((size_t)kk * p.ny + j) * NB + b) / 1.0e6;  // dmoc(:,jj,jk)/1.d6
            }
            __syncwarp();
            if (lane < NB) {
                double psi = 0.0;
                out[((size_t)nzm1 * p.ny + j) * NB + lane] = 0.0;  // dmoc(:,:,npk) stays 0
                for (int kk = nzm1 - 1; kk >= 0; --kk) {
                    psi = psi + sc[kk * NB + lane];  // dmoc(:,jj,jk+1) + dmoc(:,jj,jk)/1.d6
                    out[((size_t)kk * p.ny + j) * NB + lane] = psi;
                }
            }
            if (lane == 0) col_done[j] = 0;  // self-reset for the next launch
            __syncwarp();
        }
        u = __shfl_sync(kFull, unext, 0);
    }
}

// cdfmaxmoc epilogue (src/cdfmaxmoc.f90:158-167): extrema of REAL(psi(basin, ijmin:ijmax, ikmin:ikmax)) and their
// first location in Fortran array order, as gfortran's MAXVAL / MAXLOC (MINVAL / MINLOC) give them: NaN cells are
// skipped; the location is the first cell holding the extremum (an all -Inf window included); a window without a
// non-NaN cell gives NaN at its first cell.  One CTA of 256 threads per window w: win[5w .. 5w+4] = basin (0-based), ijmin,
// ijmax, ikmin, ikmax (1-based inclusive); res[2w ..] = max, min; loc[4w ..] = jj, jk of the max, jj, jk of the min
// (1-based).  An index of -1 means "no non-NaN cell seen" while the partial results are reduced.
__global__ void moc_window_extrema_kernel(const double *__restrict__ psi, int ny, int nb, const int32_t *__restrict__ win,
                                          float *__restrict__ res, int32_t *__restrict__ loc)
{
    __shared__ float s_max[256], s_min[256];
    __shared__ int s_imax[256], s_imin[256];
    const int32_t *w = win + 5 * blockIdx.x;
    const int basin = w[0], j0 = w[1] - 1, nj = w[2] - w[1] + 1, k0 = w[3] - 1, nk = w[4] - w[3] + 1;
    res += 2 * blockIdx.x;
    loc += 4 * blockIdx.x;
    float vmax = 0.0f, vmin = 0.0f;
    int imax = -1, imin = -1;
    for (int t = threadIdx.x; t < nj * nk; t += blockDim.x) {   // t ascends: strict comparisons keep the first location
        const int kk = t / nj, jj = t - kk * nj;
        const float v = (float)psi[((size_t)(k0 + kk) * ny + (j0 + jj)) * nb + basin];
        if (v != v) continue;
        if (imax < 0 || v > vmax) { vmax = v; imax = t; }
        if (imin < 0 || v < vmin) { vmin = v; imin = t; }
    }
    s_max[threadIdx.x] = vmax; s_imax[threadIdx.x] = imax; s_min[threadIdx.x] = vmin; s_imin[threadIdx.x] = imin;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
            const float a = s_max[threadIdx.x + o]; const int ia = s_imax[threadIdx.x + o];
            const int im = s_imax[threadIdx.x];
            if (ia >= 0 && (im < 0 || a > s_max[threadIdx.x] || (a == s_max[threadIdx.x] && ia < im))) { s_max[threadIdx.x] = a; s_imax[threadIdx.x] = ia; }
            const float b = s_min[threadIdx.x + o]; const int ib = s_imin[threadIdx.x + o];
            const int in = s_imin[threadIdx.x];
            if (ib >= 0 && (in < 0 || b < s_min[threadIdx.x] || (b == s_min[threadIdx.x] && ib < in))) { s_min[threadIdx.x] = b; s_imin[threadIdx.x] = ib; }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const bool none = s_imax[0] < 0;   // then s_imin[0] < 0 too: every cell of the window is NaN
        res[0] = none ? __int_as_float(0x7fffffff) : s_max[0];
        res[1] = none ? __int_as_float(0x7fffffff) : s_min[0];
        const int imx = none ? 0 : s_imax[0], imn = none ? 0 : s_imin[0];
        loc[0] = imx % nj + j0 + 1; loc[1] = imx / nj + k0 + 1;
        loc[2] = imn % nj + j0 + 1; loc[3] = imn / nj + k0 + 1;
    }
}

// setup kernel: area = fl32(e1v * e3m) over the n = (nz-1)*nxy cells of levels 0..nz-2; flags non-finite products.  One
// thread per flat 16-byte vector q, one warp per word of nzvec: bit q&31 of nzvec[q>>5] is set when one of the floats
// 4q..4q+3 has a non-zero bit pattern (-0.0 and NaN included; floats past n count as zero).  The block size is a multiple
// of 32 and the loop runs over whole words, so every warp reaches the ballot converged.
__global__ void moc_prep_area_kernel(const float *__restrict__ e1v, const float *__restrict__ e3m, float *__restrict__ area,
                                     uint32_t *__restrict__ nzvec, size_t nxy, size_t n, int *nonfinite)
{
    const size_t nq = (n + 127) / 128 * 32;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (size_t)gridDim.x * blockDim.x) {
        uint32_t bits = 0u;
        bool bad = false;
        size_t c = (4 * q) % nxy;
        for (int t = 0; t < 4; ++t) {
            const size_t i = 4 * q + t;
            if (i < n) {
                const float a = __fmul_rn(e1v[c], e3m[i]);
                area[i] = a;
                bits |= __float_as_uint(a);
                bad |= !isfinite(a);
            }
            if (++c == nxy) c = 0;
        }
        if (bad) atomicOr(nonfinite, 1);
        const uint32_t w = __ballot_sync(kFull, bits != 0u);
        if ((threadIdx.x & 31) == 0) nzvec[q >> 5] = w;
    }
}

}  // namespace cdfgpu
