// api.cu -- the C ABI of libcdfgpu.so (include/cdfgpu.h): context, record pipeline (pinned host buffer ->
// side-stream H2D -> fused kernel -> D2H), and the setup-time preparation of the resident mesh/mask fields.
// No CPU compute fallback exists anywhere in this file: every entry point needs a CUDA device.
#include <stdlib.h>

#include <cmath>

#include <vector>

#include "common.cuh"
#include "moc_kernel.cuh"
#include "eos_device.cuh"
#include "mocsig_kernel.cuh"
#include "moc_decomp.cuh"
#include "zonal_kernels.cuh"
#include "transig_kernels.cuh"
#include "sigtrp_kernels.cuh"
#include "unpack_kernels.cuh"
#include "microbench.cuh"

namespace cdfgpu {

char g_errbuf[512] = "";

// how one host record array is stored: REAL(4) or packed INTEGER(2) (K3b unpacks it), host order or the raw big-endian
// file bytes (K3 swap / the 16-bit swap of K3b)
struct FieldInput {
    int type = CDFGPU_INPUT_F32;
    bool big_endian = false;
    float sf = 1.f, ao = 0.f, sp = 0.f;
    size_t esize() const { return type == CDFGPU_INPUT_I16 ? sizeof(int16_t) : sizeof(float); }
};

// The declared storage of every record array, by call and field.  Rows CDFGPU_CALL_ZONAL .. _TRANSIG are the synchronous
// sibling calls (cdfgpu_set_sibling_input); row kCallSubmit holds the submit fields zv, zt, zs, zveiv, e3v_vvl of
// cdfmoc_gpu_submit, cdfmoc_gpu_decomp_submit and cdfmocsig_gpu_submit (cdfgpu_set_input_packing).  Process-wide: every
// device, until changed; cdfgpu_finalize leaves it as it is.
constexpr int kCallSubmit = CDFGPU_CALL_TRANSIG + 1, kCalls = kCallSubmit + 1, kFieldsMax = 6;
static const int kCallFields[kCalls] = {1, 2, 3, 6, 5};
// whether a row is also big-endian while cdfgpu_set_input_big_endian is on: the submits and transig are, zonal and mhst not
static const bool kCallFollowsByteOrder[kCalls] = {false, false, false, true, true};
static FieldInput g_inputs[kCalls][kFieldsMax];
static bool g_input_big_endian = false;      // cdfgpu_set_input_big_endian; cdfgpu_finalize resets it
static bool g_device_inputs_ready = false;   // cdfgpu_set_device_inputs_ready; cdfgpu_finalize resets it

// the storage a record array is copied and decoded by: as declared, and big-endian also when its row follows the flag
static FieldInput field_input(int call, int field)
{
    FieldInput in = g_inputs[call][field];
    in.big_endian = in.big_endian || (kCallFollowsByteOrder[call] && g_input_big_endian);
    return in;
}

struct Ctx {
    bool inited = false;
    int device = 0;
    int nslots = 3;
    int sm_count = 0;
    cudaStream_t s_compute = nullptr, s_copy = nullptr, s_d2h = nullptr;
    unsigned long long launches = 0;
    // latitude-band sharding (api_multi.inc): the host arrays of the current call are bands of larger arrays
    size_t host_level_stride = 0;       // elements between consecutive levels of the host record (0: contiguous)
    size_t host_out_pitch = 0;          // cdfmoc result: elements between consecutive levels of the host slab (0: contiguous)
};
constexpr int kMaxDev = 8;
static Ctx g_dev[kMaxDev];
static int g_cur = 0;      // device the single-device code below works on (the ABI is single-threaded)
static int g_ndev = 1;     // devices this process drives (cdfgpu_init: $CDFGPU_DEVICES)
static int g_shard = 0;    // 0: records go round-robin over the devices; 1: every record is split into latitude bands
static bool g_defer_sync = false;   // band gather: the per-device fetches are enqueued first and awaited together
#define g (g_dev[g_cur])

struct Workspace {  // scheduling counters of one stream-ordered sequence of launches
    int *d_tickets = nullptr;  // [3] sets of sharded counters (K1: three in rotation; the other kernels use the first two)
    int *d_col = nullptr;      // [ny]
    int parity = 0;
    int gen3 = 0;              // K1 launch generation mod 3
};

struct Slot {
    float *d_in[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // zv | zv,zt,zs,zveiv,e3v_vvl
    void *d_stage[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // raw int16 of the packed fields (n3 x 2 B)
    double *d_out = nullptr;
    cudaEvent_t ev_h2d = nullptr, ev_k0 = nullptr, ev_k1 = nullptr;
    bool used = false;
    int jt = -1;
};

// The polynomial-EOS coefficient table lives in one __constant__ symbol shared by cdfmocsig and cdfmoc -decomp; it is
// (re)loaded, stream-ordered, whenever the launching plan wants the other coefficient set.
static int g_eos_loaded_dev[kMaxDev] = {-1, -1, -1, -1, -1, -1, -1, -1};   // -1 none, 0 EOS80, 1 TEOS10 (per device)
static EosConst g_eos_host;
#define g_eos_loaded (g_eos_loaded_dev[g_cur])
static int ensure_eos(int teos10, cudaStream_t st)
{
    if (g_eos_loaded == teos10) return CDFGPU_OK;
    CDF_CUDA(cudaStreamSynchronize(st));   // g_eos_host must not be rewritten under a pending copy
    memcpy(g_eos_host.c, teos10 ? CDF_TEOS10_COEF : CDF_EOS80_COEF, sizeof(g_eos_host.c));
    memcpy(g_eos_host.r0, CDF_EOS_R0, sizeof(g_eos_host.r0));
    g_eos_host.rdeltaS = teos10 ? CDF_TEOS10_RDELTAS : CDF_EOS80_RDELTAS;
    g_eos_host.r1_S0 = teos10 ? CDF_TEOS10_R1_S0 : CDF_EOS80_R1_S0;
    CDF_CUDA(cudaDeviceSynchronize());     // no kernel of any stream may still read the old table
    CDF_CUDA(cudaMemcpyToSymbolAsync(c_eos, &g_eos_host, sizeof(g_eos_host), 0, cudaMemcpyHostToDevice, st));
    CDF_CUDA(cudaStreamSynchronize(st));
    g_eos_loaded = teos10;
    return CDFGPU_OK;
}

// host record (nlev levels of level_elems values of es bytes) -> device: contiguous, or one band of a larger array per level
static int h2d_record(void *dst, const void *src, size_t nlev, size_t level_elems, cudaStream_t st, size_t es = sizeof(float))
{
    if (g.host_level_stride == 0 || g.host_level_stride == level_elems) {
        CDF_CUDA(cudaMemcpyAsync(dst, src, nlev * level_elems * es, cudaMemcpyHostToDevice, st));
    } else {
        CDF_CUDA(cudaMemcpy2DAsync(dst, level_elems * es, src, g.host_level_stride * es, level_elems * es, nlev,
                                   cudaMemcpyHostToDevice, st));
    }
    return CDFGPU_OK;
}

static int swap_record(float *d, size_t n, cudaStream_t st, bool big_endian)
{
    if (!big_endian) return CDFGPU_OK;
    bswap32_kernel<<<g.sm_count * 8, 256, 0, st>>>(reinterpret_cast<uint32_t *>(d), n);
    CDF_CUDA(cudaGetLastError());
    ++g.launches;
    return CDFGPU_OK;
}

// H2D leg of one record field stored as `in` says: a REAL(4) record straight into d_f32, a packed one into its staging
// buffer (allocated on first use) for field_in() to decode
static int field_h2d(const FieldInput &in, float *d_f32, void *&d_stage, const float *src, size_t nlev, size_t level_elems,
                     cudaStream_t st)
{
    if (in.type == CDFGPU_INPUT_F32) return h2d_record(d_f32, src, nlev, level_elems, st);
    if (!d_stage) CDF_CUDA(cudaMalloc(&d_stage, nlev * level_elems * sizeof(int16_t) + 16));
    return h2d_record(d_stage, src, nlev, level_elems, st, sizeof(int16_t));
}

// Device leg, on the compute stream after the H2D: a packed field is unpacked from its staging buffer into d_f32 (K3b; the
// 16-bit swap when the input is big-endian), a REAL(4) field byte-swapped in place when big-endian (K3).  `fresh` becomes
// true when a kernel wrote d_f32, so that the consuming launch waits for it.
static int field_in(const FieldInput &in, float *d_f32, const void *d_stage, size_t n, cudaStream_t st, bool &fresh)
{
    if (in.type == CDFGPU_INPUT_F32) {
        fresh = fresh || in.big_endian;
        return swap_record(d_f32, n, st, in.big_endian);
    }
    const int grid = (int)std::min<size_t>((size_t)g.sm_count * 8, std::max<size_t>((n / 8 + 255) / 256, 1));
    unpack_i16_kernel<<<grid, 256, 0, st>>>(static_cast<const uint16_t *>(d_stage), d_f32, n, in.big_endian ? 1 : 0, in.sf,
                                            in.ao, in.sp);
    CDF_CUDA(cudaGetLastError());
    ++g.launches;
    fresh = true;
    return CDFGPU_OK;
}

// Both legs of one record array (nlev levels of level_elems values) on the one stream st, stored as field_input(call, field)
// says: the synchronous sibling calls, and -decomp's T and S, whose consumers follow on the same stream.
static int field_h2d_in(int call, int field, float *d_f32, void *&d_stage, const float *src, size_t nlev, size_t level_elems,
                        cudaStream_t st)
{
    const FieldInput in = field_input(call, field);
    bool fresh = false;
    const int rc = field_h2d(in, d_f32, d_stage, src, nlev, level_elems, st);
    return rc ? rc : field_in(in, d_f32, d_stage, nlev * level_elems, st, fresh);
}

static int make_ws(Workspace &w, int ny)
{
    CDF_CUDA(cudaMalloc(&w.d_tickets, 3 * kTicketShards * kTicketStride * sizeof(int)));
    CDF_CUDA(cudaMalloc(&w.d_col, (size_t)ny * sizeof(int)));
    CDF_CUDA(cudaMemsetAsync(w.d_tickets, 0, 3 * kTicketShards * kTicketStride * sizeof(int), g.s_compute));
    CDF_CUDA(cudaMemsetAsync(w.d_col, 0, (size_t)ny * sizeof(int), g.s_compute));
    w.parity = 0;
    w.gen3 = 0;
    return CDFGPU_OK;
}
static void free_ws(Workspace &w)
{
    cudaFree(w.d_tickets);
    cudaFree(w.d_col);
    w = Workspace();
}
static int make_slot_events(Slot &s)
{
    CDF_CUDA(cudaEventCreateWithFlags(&s.ev_h2d, cudaEventDisableTiming));
    CDF_CUDA(cudaEventCreate(&s.ev_k0));
    CDF_CUDA(cudaEventCreate(&s.ev_k1));
    return CDFGPU_OK;
}
static void free_slot(Slot &s)
{
    for (auto &p : s.d_in) cudaFree(p);
    for (auto &p : s.d_stage) cudaFree(p);
    cudaFree(s.d_out);
    if (s.ev_h2d) cudaEventDestroy(s.ev_h2d);
    if (s.ev_k0) cudaEventDestroy(s.ev_k0);
    if (s.ev_k1) cudaEventDestroy(s.ev_k1);
    s = Slot();
}

// Packs (nb,nx,ny) INTEGER(2) masks into one byte per cell and builds the 4 pre-shifted word planes.
// Returns false if some mask value is not 0/1 (then only the general path is valid).
static bool pack_masks(int nx, int ny, int nb, const int16_t *ibmask, int pitchw, std::vector<uint32_t> &words)
{
    bool binary = true;
    std::vector<uint8_t> bits((size_t)nx * ny);
    for (size_t c = 0; c < (size_t)nx * ny; ++c) {
        uint8_t v = 0;
        for (int b = 0; b < nb; ++b) {
            const int16_t m = ibmask[c * nb + b];
            if (m != 0 && m != 1) binary = false;
            if (m != 0) v |= (uint8_t)(1u << b);
        }
        bits[c] = v;
    }
    words.assign((size_t)4 * ny * pitchw, 0u);
    for (int s = 0; s < 4; ++s)
        for (int j = 0; j < ny; ++j) {
            uint32_t *row = words.data() + ((size_t)s * ny + j) * pitchw;
            const uint8_t *brow = bits.data() + (size_t)j * nx;
            for (int w = 0; w < pitchw; ++w) {
                uint32_t x = 0;
                for (int c = 0; c < 4; ++c) {
                    const long i = 4L * w - s + c;
                    if (i >= 0 && i < nx) x |= (uint32_t)brow[i] << (8 * c);
                }
                row[w] = x;
            }
        }
    return binary;
}

// =================================================================================================== cdfmoc
struct MocPlan {
    bool ready = false;
    int nx = 0, ny = 0, nz = 0, nb = 0, pitchw = 0, general = 0, general_masks = 0, chunk = 1, jsplit = 0;
    float *d_e1v = nullptr, *d_e3m = nullptr, *d_area = nullptr;
    uint32_t *d_maskw = nullptr;
    uint32_t *d_nzvec = nullptr;   // one bit per 16-byte vector of d_area: 1 = not all four words are +0.0f
    int16_t *d_ibmask = nullptr;
    int *d_flag = nullptr;
    float *d_ext = nullptr;   // cdfmaxmoc epilogue result
    // -decomp (cdfmoc.f90:390-517)
    bool decomp = false;
    int dec_teos10 = 0;
    int dec_pending = -1;   // slot whose decomposition has been submitted and not fetched yet
    float *d_e1u = nullptr, *d_zcoef = nullptr, *d_zt = nullptr, *d_zs = nullptr, *d_sig = nullptr, *d_hdep = nullptr,
          *d_zvgeo = nullptr;
    int16_t *d_umask = nullptr, *d_tmask = nullptr;
    double *d_dvbt = nullptr, *d_dvgeo = nullptr, *d_sh = nullptr, *d_bt = nullptr, *d_ag = nullptr, *d_btw = nullptr;
    std::vector<double> dec_dlh, dec_dlref;
    Workspace ws_int, ws_ext;
    Slot slots[CDFGPU_MAX_SLOTS];
    int grid = 0, grid_batch = 0;
    size_t smem = 0;
    bool pdl = true;       // programmatic dependent launch ($CDFGPU_K1_PDL=0 switches it off)
    // batched launches (cdfmoc_gpu_compute_device_batch): device arrays of record / slab pointers, column counters
    const float **d_batch_zv = nullptr;
    double **d_batch_out = nullptr;
    int *d_batch_col = nullptr;
    int batch_cap = 0, batch_flip = 0;
    size_t in_elems() const { return (size_t)(nz - 1) * ny * nx; }
    size_t out_elems() const { return (size_t)nz * ny * nb; }
};
static MocPlan moc_dev[kMaxDev];
#define moc (moc_dev[g_cur])

template <int NB, int UNROLL, int MINB, bool BATCH>
static int moc_launch_v(const MocParams &p, cudaStream_t st)
{
    auto kern = moc_zonal_scan_kernel<NB, UNROLL, MINB, BATCH>;
    int &grid = BATCH ? moc.grid_batch : moc.grid;
    if (grid == 0) {
        int occ = 0;
        CDF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)moc.smem));
        CDF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kMocThreads, moc.smem));
        if (occ < 1) return set_error(CDFGPU_ERR_ARG, "cdfmoc: kernel does not fit (nz*nb too large for shared memory)");
        // $CDFGPU_K1_SPARE_SMS: leave a few SMs to kernels of other streams (an NCCL slab gather running beside the
        // persistent grid otherwise takes its SMs from it at the launch boundaries)
        int spare = 0;
        if (const char *e = getenv("CDFGPU_K1_SPARE_SMS")) spare = std::max(0, std::min(g.sm_count - 1, atoi(e)));
        grid = occ * (g.sm_count - spare);
    }
    if (moc.pdl) {   // programmatic dependent launch: consecutive K1 launches of a stream overlap tail and ramp-up
        MocParams q = p;
        q.pdl = 1;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3(kMocThreads);
        cfg.dynamicSmemBytes = moc.smem;
        cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        CDF_CUDA(cudaLaunchKernelEx(&cfg, kern, q));
    } else {
        kern<<<grid, kMocThreads, moc.smem, st>>>(p);
    }
    CDF_CUDA(cudaGetLastError());
    ++g.launches;
    return CDFGPU_OK;
}
template <int NB>
static int moc_launch_t(const MocParams &p, cudaStream_t st)
{
    // 4 vector pairs per lane in flight, 3 CTAs of 256 threads per SM.  The staged feeds (cp.async / TMA rings), the class
    // formulation and the other unroll / occupancy points measured in round 1 (profiles/r01_k1_*.{txt,json}) were all
    // slower and are no longer built; their sources are in the history (moc_kernel_{pipe,tma,class}.cuh at 028f76b).
    return p.nrec > 1 ? moc_launch_v<NB, 4, 3, true>(p, st) : moc_launch_v<NB, 4, 3, false>(p, st);
}

// inputs_fresh: the record (or the area field) may have been written by work enqueued on `st` after the previous K1 launch
// (byte swap, -vvl area build, -decomp stencil, a caller's producer kernel): no load may then precede griddepcontrol.wait.
// nrec > 1: one launch over the records zv_list[0..nrec) -> out_list[0..nrec) (device arrays of pointers).
static int moc_launch(const float *d_zv, double *d_out, Workspace &ws, cudaStream_t st, int noscan = 0, bool inputs_fresh = true,
                      int nrec = 1, const float *const *zv_list = nullptr, double *const *out_list = nullptr, int *batch_col = nullptr)
{
    MocParams p;
    p.zv = d_zv;
    p.area = moc.d_area;
    p.nzvec = moc.d_nzvec;
    p.maskw = moc.d_maskw;
    p.ibmask = moc.d_ibmask;
    p.out = d_out;
    p.tickets = ws.d_tickets;
    p.col_done = batch_col ? batch_col : ws.d_col;
    p.nx = moc.nx; p.ny = moc.ny; p.nz = moc.nz; p.pitchw = moc.pitchw;
    p.parity = ws.gen3;
    ws.gen3 = (ws.gen3 + 1) % 3;
    p.pdl = 0;
    p.pdl_early = inputs_fresh ? 0 : 1;
    p.chunk = moc.chunk;
    p.jsplit = moc.jsplit;
    p.general = moc.general;
    p.noscan = noscan;
    p.nrec = nrec;
    p.zv_list = zv_list;
    p.out_list = out_list;
    ws.parity ^= 1;
    switch (moc.nb) {
    case 1: return moc_launch_t<1>(p, st);
    case 2: return moc_launch_t<2>(p, st);
    case 3: return moc_launch_t<3>(p, st);
    case 4: return moc_launch_t<4>(p, st);
    case 5: return moc_launch_t<5>(p, st);
    case 6: return moc_launch_t<6>(p, st);
    case 7: return moc_launch_t<7>(p, st);
    case 8: return moc_launch_t<8>(p, st);
    }
    return set_error(CDFGPU_ERR_ARG, "cdfmoc: nb must be 1..8");
}

static int moc_build_area()
{
    const size_t nxy = (size_t)moc.nx * moc.ny, n = moc.in_elems();
    CDF_CUDA(cudaMemsetAsync(moc.d_flag, 0, sizeof(int), g.s_compute));
    const unsigned grid = (unsigned)std::min<size_t>((n + 1023) / 1024, (size_t)g.sm_count * 8);
    moc_prep_area_kernel<<<grid, 256, 0, g.s_compute>>>(moc.d_e1v, moc.d_e3m, moc.d_area, moc.d_nzvec, nxy, n, moc.d_flag);
    CDF_CUDA(cudaGetLastError());
    ++g.launches;
    int flag = 0;
    CDF_CUDA(cudaMemcpyAsync(&flag, moc.d_flag, sizeof(int), cudaMemcpyDeviceToHost, g.s_compute));
    CDF_CUDA(cudaStreamSynchronize(g.s_compute));
    moc.general = (moc.general_masks || flag) ? 1 : 0;   // (a later -vvl record with a finite area takes the fast path again)
    return CDFGPU_OK;
}

template <int NB>
static void decomp_weighted_t(const double *w, double *raw, cudaStream_t st)
{
    decomp_weighted_rows_kernel<NB><<<g.sm_count * 4, 256, 0, st>>>(moc.d_area, moc.d_ibmask, w, moc.nx, moc.ny, moc.nz - 1, raw);
}
static int decomp_weighted(const double *w, double *raw, cudaStream_t st)
{
    switch (moc.nb) {
    case 1: decomp_weighted_t<1>(w, raw, st); break;
    case 2: decomp_weighted_t<2>(w, raw, st); break;
    case 3: decomp_weighted_t<3>(w, raw, st); break;
    case 4: decomp_weighted_t<4>(w, raw, st); break;
    case 5: decomp_weighted_t<5>(w, raw, st); break;
    case 6: decomp_weighted_t<6>(w, raw, st); break;
    case 7: decomp_weighted_t<7>(w, raw, st); break;
    default: decomp_weighted_t<8>(w, raw, st); break;
    }
    CDF_CUDA(cudaGetLastError());
    ++g.launches;
    return CDFGPU_OK;
}

}  // namespace cdfgpu

using namespace cdfgpu;

#define REQUIRE_INIT()                                                                           \
    if (!g.inited) return set_error(CDFGPU_ERR_STATE, "cdfgpu_init has not been called")
#define REQUIRE(cond, code, msg)                                                                 \
    if (!(cond)) return set_error(code, msg)
// the synchronous sibling calls (cdfzonal*, cdfmhst, cdftransig, cdfsigtrp) and the probes run on the first device of the process
#define FIRST_DEVICE()                                  \
    do {                                                \
        if (g_cur != 0) {                               \
            g_cur = 0;                                  \
            cudaSetDevice(g_dev[0].device);             \
        }                                               \
    } while (0)
// the entry points that take device pointers (*_device): those belong to one device
static int single_device_only(const char *what)
{
    if (g_ndev > 1)
        return set_error(CDFGPU_ERR_STATE, "%s: device pointers belong to one device -- drive it with one process per GPU "
                                           "(CDFGPU_DEVICES unset)", what);
    return CDFGPU_OK;
}
#define SINGLE_DEVICE_ONLY(what) \
    if (int rc__ = single_device_only(what)) return rc__

extern "C" {
static int cdfmoc_gpu_teardown_dev(void);
static int cdfmocsig_gpu_teardown_dev(void);
static int cdfzonal_gpu_teardown_dev(void);
static int cdfmhst_gpu_teardown_dev(void);
static int cdftransig_gpu_teardown_dev(void);
static int cdfmocsig_gpu_bins_device_stats_dev(const float *d_zt, const float *d_zs, int32_t *d_ibin, unsigned long long *stats3, void *stream);

int cdfgpu_abi_version(void) { return 1; }

const char *cdfgpu_strerror(int code)
{
    switch (code) {
    case CDFGPU_OK: return "ok";
    case CDFGPU_ERR_CUDA: return "CUDA runtime error";
    case CDFGPU_ERR_ARG: return "invalid argument";
    case CDFGPU_ERR_STATE: return "call order violated";
    case CDFGPU_ERR_NOMEM: return "out of device or pinned memory";
    case CDFGPU_ERR_NODEVICE: return "no CUDA device available (libcdfgpu has no CPU fallback)";
    }
    return "unknown error";
}
const char *cdfgpu_last_error(void) { return g_errbuf; }

int cdfgpu_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        set_error(CDFGPU_ERR_NODEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
        cudaGetLastError();
        return -CDFGPU_ERR_NODEVICE;
    }
    return n;
}

static int cdfgpu_init_dev(int device, int nslots)
{
    if (g.inited) return CDFGPU_OK;
    const int n = cdfgpu_device_count();
    if (n <= 0) {
        char why[256];
        snprintf(why, sizeof(why), "%.200s", n < 0 ? g_errbuf : "device count is 0");
        return set_error(CDFGPU_ERR_NODEVICE, "no CUDA device visible: %s", why);
    }
    if (device < 0) {
        const char *e = getenv("CDFGPU_DEVICE");
        device = e ? atoi(e) : 0;
    }
    REQUIRE(device < n, CDFGPU_ERR_ARG, "cdfgpu_init: device ordinal out of range");
    if (nslots == 0) {
        const char *e = getenv("CDFGPU_SLOTS");
        nslots = e ? atoi(e) : 3;
    }
    REQUIRE(nslots >= 1 && nslots <= CDFGPU_MAX_SLOTS, CDFGPU_ERR_ARG, "cdfgpu_init: nslots must be 1..8");
    CDF_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    CDF_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return set_error(CDFGPU_ERR_NODEVICE, "libcdfgpu is built for sm_100a only; device is %s", prop.name);
    g.device = device;
    g.nslots = nslots;
    g.sm_count = prop.multiProcessorCount;
    CDF_CUDA(cudaStreamCreateWithFlags(&g.s_compute, cudaStreamNonBlocking));
    CDF_CUDA(cudaStreamCreateWithFlags(&g.s_copy, cudaStreamNonBlocking));
    CDF_CUDA(cudaStreamCreateWithFlags(&g.s_d2h, cudaStreamNonBlocking));
    g.launches = 0;
    g.inited = true;
    return CDFGPU_OK;
}

static int cdfgpu_synchronize_dev(void)
{
    REQUIRE_INIT();
    CDF_CUDA(cudaStreamSynchronize(g.s_copy));
    CDF_CUDA(cudaStreamSynchronize(g.s_compute));
    CDF_CUDA(cudaStreamSynchronize(g.s_d2h));
    return CDFGPU_OK;
}

static int cdfgpu_finalize_dev(void)
{
    if (!g.inited) return CDFGPU_OK;
    cdfgpu_synchronize_dev();
    cdfmoc_gpu_teardown_dev();
    cdfmocsig_gpu_teardown_dev();
    cdfzonal_gpu_teardown_dev();
    cdfmhst_gpu_teardown_dev();
    cdftransig_gpu_teardown_dev();
    if (g_cur == 0) cdfsigtrp_gpu_teardown();   // cdfsigtrp lives on the first device
    cudaStreamDestroy(g.s_compute);
    cudaStreamDestroy(g.s_copy);
    cudaStreamDestroy(g.s_d2h);
    g = Ctx();
    g_eos_loaded = -1;
    cudaGetLastError();   // nothing left pending for the next session of this process
    return CDFGPU_OK;
}

void *cdfgpu_pinned_alloc(size_t nbytes)
{
    void *p = nullptr;
    cudaError_t e = cudaHostAlloc(&p, nbytes ? nbytes : 1, cudaHostAllocPortable);   // page-locked for every device of the process
    if (e != cudaSuccess) {
        set_error(CDFGPU_ERR_NOMEM, "cudaHostAlloc: %s", cudaGetErrorString(e));
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
int cdfgpu_pinned_free(void *p)
{
    if (p) CDF_CUDA(cudaFreeHost(p));
    return CDFGPU_OK;
}
// Platform ceiling of the record pipeline's input leg: `reps` asynchronous copies of a pinned host buffer to device memory
// on the library's copy stream, nothing else running.  gbs = GB/s of this process (bench.py sums the ranks).
int cdfgpu_h2d_probe(const void *pinned, size_t nbytes, int reps, double *gbs)
{
    FIRST_DEVICE();
    REQUIRE_INIT();
    REQUIRE(pinned && nbytes > 0 && reps > 0 && gbs, CDFGPU_ERR_ARG, "cdfgpu_h2d_probe: bad argument");
    void *d = nullptr;
    CDF_CUDA(cudaMalloc(&d, nbytes));
    cudaEvent_t e0, e1;
    CDF_CUDA(cudaEventCreate(&e0));
    CDF_CUDA(cudaEventCreate(&e1));
    CDF_CUDA(cudaMemcpyAsync(d, pinned, nbytes, cudaMemcpyHostToDevice, g.s_copy));   // warm-up
    CDF_CUDA(cudaEventRecord(e0, g.s_copy));
    for (int r = 0; r < reps; ++r) CDF_CUDA(cudaMemcpyAsync(d, pinned, nbytes, cudaMemcpyHostToDevice, g.s_copy));
    CDF_CUDA(cudaEventRecord(e1, g.s_copy));
    CDF_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    CDF_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    *gbs = (double)nbytes * reps / (ms * 1e-3) / 1e9;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(d);
    return CDFGPU_OK;
}
unsigned long long cdfgpu_launch_count(void)
{
    unsigned long long n = 0;
    for (int d = 0; d < g_ndev; ++d) n += g_dev[d].launches;
    return n;
}
int cdfgpu_set_input_big_endian(int on)
{
    g_input_big_endian = on != 0;
    return CDFGPU_OK;
}

// kind: 0 DFMA, 1 FFMA, 2 FFMA2 (packed fp32), 3 integer (LOP3 + shift-add), 4 FFMA alternating with integer operations.
// out[0] = warp-instructions per clock and SM (the slowest CTA's own clock64 window), out[1] = 1e9 warp-instructions / s
// over the chip (CUDA events), out[2] = SM clock in MHz implied by the two.
int cdfgpu_microbench(int kind, double *out3)
{
    FIRST_DEVICE();
    REQUIRE_INIT();
    REQUIRE(kind >= 0 && kind <= 4 && out3, CDFGPU_ERR_ARG, "cdfgpu_microbench: kind must be 0..4");
    const int iters = 20000, nblk = g.sm_count;
    unsigned long long *d_cyc = nullptr;
    double *d_sink = nullptr;
    CDF_CUDA(cudaMalloc(&d_cyc, nblk * sizeof(unsigned long long)));
    CDF_CUDA(cudaMalloc(&d_sink, sizeof(double)));
    cudaEvent_t e0, e1;
    CDF_CUDA(cudaEventCreate(&e0));
    CDF_CUDA(cudaEventCreate(&e1));
    float ms = 0.f;
    for (int rep = 0; rep < 2; ++rep) {   // first pass warms up
        CDF_CUDA(cudaEventRecord(e0, g.s_compute));
        switch (kind) {
        case kMbDfma: microbench_kernel<kMbDfma><<<nblk, 1024, 0, g.s_compute>>>(iters, 1.0f, d_cyc, d_sink); break;
        case kMbFfma: microbench_kernel<kMbFfma><<<nblk, 1024, 0, g.s_compute>>>(iters, 1.0f, d_cyc, d_sink); break;
        case kMbFfma2: microbench_kernel<kMbFfma2><<<nblk, 1024, 0, g.s_compute>>>(iters, 1.0f, d_cyc, d_sink); break;
        case kMbIadd: microbench_kernel<kMbIadd><<<nblk, 1024, 0, g.s_compute>>>(iters, 1.0f, d_cyc, d_sink); break;
        default: microbench_kernel<kMbMixed><<<nblk, 1024, 0, g.s_compute>>>(iters, 1.0f, d_cyc, d_sink); break;
        }
        CDF_CUDA(cudaGetLastError());
        ++g.launches;
        CDF_CUDA(cudaEventRecord(e1, g.s_compute));
        CDF_CUDA(cudaEventSynchronize(e1));
        CDF_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    }
    std::vector<unsigned long long> cyc(nblk);
    CDF_CUDA(cudaMemcpy(cyc.data(), d_cyc, nblk * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    unsigned long long mx = 1;
    for (auto c : cyc) mx = std::max(mx, c);
    // per trip: kinds 0..2 issue 32 operations, kind 3 issues 64 (two per step), kind 4 issues 48 (fma + xor + add per step)
    const double per_trip = kind == kMbIadd ? 64.0 : kind == kMbMixed ? 48.0 : 32.0;
    const double winst_per_sm = (double)iters * per_trip * 32.0;   // 32 warps per CTA
    out3[0] = winst_per_sm / (double)mx;
    out3[1] = winst_per_sm * nblk / (ms * 1e-3) / 1e9;
    out3[2] = (double)mx / (ms * 1e-3) / 1e6;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(d_cyc); cudaFree(d_sink);
    return CDFGPU_OK;
}

// stores the declaration of g_inputs[call][field] (the caller has checked the indices); `setter` names the entry point in
// the error messages
static int set_field_input(const char *setter, int call, int field, int type, bool big_endian, float scale_factor,
                           float add_offset, float spval)
{
    if (type != CDFGPU_INPUT_F32 && type != CDFGPU_INPUT_I16)
        return set_error(CDFGPU_ERR_ARG, "%s: type must be CDFGPU_INPUT_F32 or CDFGPU_INPUT_I16", setter);
    if (type == CDFGPU_INPUT_I16 && !(std::isfinite(scale_factor) && std::isfinite(add_offset)))
        return set_error(CDFGPU_ERR_ARG, "%s: scale_factor and add_offset must be finite", setter);
    FieldInput in;
    in.big_endian = big_endian;
    if (type == CDFGPU_INPUT_I16) {
        in.type = type;
        in.sf = scale_factor; in.ao = add_offset; in.sp = spval;
    }
    g_inputs[call][field] = in;
    return CDFGPU_OK;
}

int cdfgpu_set_input_packing(int field, int type, float scale_factor, float add_offset, float spval)
{
    REQUIRE(field >= 0 && field < kCallFields[kCallSubmit], CDFGPU_ERR_ARG,
            "cdfgpu_set_input_packing: field must be 0..4 (zv, zt, zs, zveiv, e3v_vvl)");
    return set_field_input("cdfgpu_set_input_packing", kCallSubmit, field, type, false, scale_factor, add_offset, spval);
}

int cdfgpu_set_sibling_input(int call, int field, int type, int big_endian, float scale_factor, float add_offset, float spval)
{
    REQUIRE(call >= 0 && call < kCallSubmit, CDFGPU_ERR_ARG,
            "cdfgpu_set_sibling_input: call must be CDFGPU_CALL_ZONAL, _MHST, _MHST_VTS or _TRANSIG");
    REQUIRE(field >= 0 && field < kCallFields[call], CDFGPU_ERR_ARG,
            "cdfgpu_set_sibling_input: field outside the call's arrays (zonal: 0 zv; mhst: 0 zvt, 1 zvs; mhst_vts: 0 zv, 1 zt, "
            "2 zs; transig: 0 zu, 1 zv, 2 zt, 3 zs, 4 e3u_vvl, 5 e3v_vvl)");
    return set_field_input("cdfgpu_set_sibling_input", call, field, type, big_endian != 0, scale_factor, add_offset, spval);
}

int cdfgpu_set_device_inputs_ready(int on)
{
    g_device_inputs_ready = on != 0;
    return CDFGPU_OK;
}

// --------------------------------------------------------------------------------------------------- cdfmoc
static int cdfmoc_gpu_teardown_dev(void)
{
    if (!moc.ready && !moc.d_area) return CDFGPU_OK;
    if (g.inited) cdfgpu_synchronize_dev();
    cudaFree(moc.d_e1v); cudaFree(moc.d_e3m); cudaFree(moc.d_area); cudaFree(moc.d_nzvec); cudaFree(moc.d_maskw);
    cudaFree(moc.d_ibmask); cudaFree(moc.d_flag); cudaFree(moc.d_ext);
    cudaFree(moc.d_batch_zv); cudaFree(moc.d_batch_out); cudaFree(moc.d_batch_col);
    cudaFree(moc.d_e1u); cudaFree(moc.d_zcoef); cudaFree(moc.d_zt); cudaFree(moc.d_zs); cudaFree(moc.d_sig);
    cudaFree(moc.d_hdep); cudaFree(moc.d_zvgeo); cudaFree(moc.d_umask); cudaFree(moc.d_tmask); cudaFree(moc.d_dvbt);
    cudaFree(moc.d_dvgeo); cudaFree(moc.d_sh); cudaFree(moc.d_bt); cudaFree(moc.d_ag); cudaFree(moc.d_btw);
    free_ws(moc.ws_int); free_ws(moc.ws_ext);
    for (auto &s : moc.slots) free_slot(s);
    moc = MocPlan();
    return CDFGPU_OK;
}

static int cdfmoc_gpu_setup_dev(int nx, int ny, int nz, int nb, const float *e1v, const float *e3v, const int16_t *ibmask)
{
    REQUIRE_INIT();
    REQUIRE(nx >= 1 && ny >= 1 && nz >= 2, CDFGPU_ERR_ARG, "cdfmoc_gpu_setup: need nx,ny >= 1 and nz >= 2");
    REQUIRE(nb >= 1 && nb <= CDFGPU_MAX_BASINS, CDFGPU_ERR_ARG, "cdfmoc_gpu_setup: nb must be 1..8");
    REQUIRE(e1v && e3v && ibmask, CDFGPU_ERR_ARG, "cdfmoc_gpu_setup: null pointer");
    REQUIRE((size_t)nx * ny * (nz - 1) / 4 < ((size_t)1 << 32), CDFGPU_ERR_ARG,
            "cdfmoc_gpu_setup: more than 2^34 cells per record (K1 indexes 16-byte vectors with 32 bits)");
    cdfmoc_gpu_teardown_dev();
    moc.nx = nx; moc.ny = ny; moc.nz = nz; moc.nb = nb;
    moc.pitchw = ((nx + 6) / 4 + 1 + 3) & ~3;   // rows of the mask planes start on 16-byte boundaries (bulk copies)
    {
        const char *d = getenv("CDFGPU_K1_PDL");
        moc.pdl = !(d && atoi(d) == 0);
    }
    // rows shorter than ~16 KB are handed out several levels at a time: fewer tickets, fences and column counters
    moc.chunk = (nx < 4096) ? 4 : 1;   // levels per work unit (ORCA025: 4 -> 5.49 TB/s, 2 -> 5.39, 1 -> 5.14)
    if (const char *c = getenv("CDFGPU_K1_CHUNK")) moc.chunk = std::max(1, atoi(c));
    {   // optional guided hand-out: the last 1/den of the columns one level per ticket (a shorter tail of the launch).
        // Measured neutral on ORCA025 (0.158-0.164 ms for den = 0, 16, 8, 4, 2): off by default; $CDFGPU_K1_TAIL = den
        int den = 0;
        if (const char *c = getenv("CDFGPU_K1_TAIL")) den = atoi(c);
        moc.jsplit = (moc.chunk > 1 && den > 0) ? ny - ny / den : ny;
    }
    const size_t nxy = (size_t)nx * ny;
    CDF_CUDA(cudaMalloc(&moc.d_e1v, nxy * sizeof(float)));
    CDF_CUDA(cudaMalloc(&moc.d_e3m, nxy * (size_t)(nz - 1) * sizeof(float)));
    CDF_CUDA(cudaMalloc(&moc.d_area, nxy * (size_t)(nz - 1) * sizeof(float) + 16));
    // the last vector of the area array reaches into the 16-byte pad: zeros there, as the bitmap assumes
    CDF_CUDA(cudaMemsetAsync(moc.d_area + nxy * (size_t)(nz - 1), 0, 16, g.s_compute));
    CDF_CUDA(cudaMalloc(&moc.d_nzvec, (nxy * (size_t)(nz - 1) + 127) / 128 * sizeof(uint32_t)));
    CDF_CUDA(cudaMalloc(&moc.d_ibmask, nxy * nb * sizeof(int16_t)));
    CDF_CUDA(cudaMalloc(&moc.d_maskw, (size_t)4 * ny * moc.pitchw * sizeof(uint32_t)));
    CDF_CUDA(cudaMalloc(&moc.d_flag, sizeof(int)));
    int rc;
    if ((rc = make_ws(moc.ws_int, ny))) return rc;
    if ((rc = make_ws(moc.ws_ext, ny))) return rc;
    std::vector<uint32_t> words;
    const bool binary = pack_masks(nx, ny, nb, ibmask, moc.pitchw, words);
    moc.general_masks = binary ? 0 : 1;
    moc.general = moc.general_masks;
    CDF_CUDA(cudaMemcpyAsync(moc.d_maskw, words.data(), words.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, g.s_compute));
    CDF_CUDA(cudaMemcpyAsync(moc.d_ibmask, ibmask, nxy * nb * sizeof(int16_t), cudaMemcpyHostToDevice, g.s_compute));
    CDF_CUDA(cudaMemcpyAsync(moc.d_e1v, e1v, nxy * sizeof(float), cudaMemcpyHostToDevice, g.s_compute));
    CDF_CUDA(cudaMemcpyAsync(moc.d_e3m, e3v, nxy * (size_t)(nz - 1) * sizeof(float), cudaMemcpyHostToDevice, g.s_compute));
    if ((rc = moc_build_area())) return rc;
    moc.smem = (size_t)(kMocThreads / 32) * (nz - 1) * nb * sizeof(double);
    moc.grid = 0;
    moc.grid_batch = 0;
    for (int s = 0; s < g.nslots; ++s) {
        if ((rc = make_slot_events(moc.slots[s]))) return rc;
        CDF_CUDA(cudaMalloc(&moc.slots[s].d_in[0], moc.in_elems() * sizeof(float) + 16));
        CDF_CUDA(cudaMalloc(&moc.slots[s].d_out, moc.out_elems() * sizeof(double)));
    }
    CDF_CUDA(cudaStreamSynchronize(g.s_compute));  // setup copies are ordered on the compute stream; drain them
    moc.ready = true;
    return CDFGPU_OK;
}

static int cdfmoc_gpu_set_e3v_dev(const float *e3v)
{
    REQUIRE_INIT();
    REQUIRE(moc.ready, CDFGPU_ERR_STATE, "cdfmoc_gpu_set_e3v: cdfmoc_gpu_setup has not been called");
    REQUIRE(e3v, CDFGPU_ERR_ARG, "cdfmoc_gpu_set_e3v: null pointer");
    // the area field is read by every kernel in flight: drain first (rare path, once per record with -vvl)
    CDF_CUDA(cudaStreamSynchronize(g.s_compute));
    CDF_CUDA(cudaMemcpyAsync(moc.d_e3m, e3v, (size_t)moc.nx * moc.ny * (moc.nz - 1) * sizeof(float), cudaMemcpyHostToDevice, g.s_compute));
    return moc_build_area();
}

static int cdfmoc_gpu_submit_dev(int slot, int jt, const float *zv)
{
    REQUIRE_INIT();
    REQUIRE(moc.ready, CDFGPU_ERR_STATE, "cdfmoc_gpu_submit: cdfmoc_gpu_setup has not been called");
    REQUIRE(slot >= 0 && slot < g.nslots, CDFGPU_ERR_ARG, "cdfmoc_gpu_submit: slot out of range");
    REQUIRE(zv, CDFGPU_ERR_ARG, "cdfmoc_gpu_submit: null pointer");
    Slot &s = moc.slots[slot];
    const FieldInput in = field_input(kCallSubmit, 0);
    if (s.used) CDF_CUDA(cudaStreamWaitEvent(g.s_copy, s.ev_k1, 0));  // previous kernel on this slot has read d_in
    {
        int rch = field_h2d(in, s.d_in[0], s.d_stage[0], zv, (size_t)(moc.nz - 1), (size_t)moc.ny * moc.nx, g.s_copy);
        if (rch) return rch;
    }
    CDF_CUDA(cudaEventRecord(s.ev_h2d, g.s_copy));
    CDF_CUDA(cudaStreamWaitEvent(g.s_compute, s.ev_h2d, 0));
    bool fresh = false;
    int rc = field_in(in, s.d_in[0], s.d_stage[0], moc.in_elems(), g.s_compute, fresh);
    if (rc) return rc;
    CDF_CUDA(cudaEventRecord(s.ev_k0, g.s_compute));
    // the H2D copy is ordered by the event above; a byte swap or an unpack on this stream writes the record right before K1
    rc = moc_launch(s.d_in[0], s.d_out, moc.ws_int, g.s_compute, 0, fresh);
    if (rc) return rc;
    CDF_CUDA(cudaEventRecord(s.ev_k1, g.s_compute));
    s.used = true;
    s.jt = jt;
    return CDFGPU_OK;
}

static int cdfmoc_gpu_fetch_dev(int slot, double *dmoc)
{
    REQUIRE_INIT();
    REQUIRE(moc.ready, CDFGPU_ERR_STATE, "cdfmoc_gpu_fetch: cdfmoc_gpu_setup has not been called");
    REQUIRE(slot >= 0 && slot < g.nslots, CDFGPU_ERR_ARG, "cdfmoc_gpu_fetch: slot out of range");
    REQUIRE(dmoc, CDFGPU_ERR_ARG, "cdfmoc_gpu_fetch: null pointer");
    Slot &s = moc.slots[slot];
    REQUIRE(s.used, CDFGPU_ERR_STATE, "cdfmoc_gpu_fetch: nothing was submitted on this slot");
    CDF_CUDA(cudaStreamWaitEvent(g.s_d2h, s.ev_k1, 0));
    const size_t lev = (size_t)moc.ny * moc.nb;   // one level of the slab: (ny, nb)
    if (g.host_out_pitch == 0 || g.host_out_pitch == lev) {
        CDF_CUDA(cudaMemcpyAsync(dmoc, s.d_out, moc.out_elems() * sizeof(double), cudaMemcpyDeviceToHost, g.s_d2h));
    } else {
        CDF_CUDA(cudaMemcpy2DAsync(dmoc, g.host_out_pitch * sizeof(double), s.d_out, lev * sizeof(double), lev * sizeof(double),
                                   (size_t)moc.nz, cudaMemcpyDeviceToHost, g.s_d2h));
    }
    if (!g_defer_sync) CDF_CUDA(cudaStreamSynchronize(g.s_d2h));
    return CDFGPU_OK;
}

static int cdfmoc_gpu_compute_device_dev(const float *d_zv, double *d_dmoc, void *stream)
{
    REQUIRE_INIT();
    REQUIRE(moc.ready, CDFGPU_ERR_STATE, "cdfmoc_gpu_compute_device: cdfmoc_gpu_setup has not been called");
    REQUIRE(d_zv && d_dmoc, CDFGPU_ERR_ARG, "cdfmoc_gpu_compute_device: null pointer");
    // on the library's own stream the caller must have synchronised its producers; on a caller stream the record may come
    // from the kernel right before this one unless the caller said otherwise (cdfgpu_set_device_inputs_ready)
    if (stream == nullptr) return moc_launch(d_zv, d_dmoc, moc.ws_int, g.s_compute, 0, false);
    return moc_launch(d_zv, d_dmoc, moc.ws_ext, (cudaStream_t)stream, 0, !g_device_inputs_ready);
}

// One launch over nrec device-resident records: the work units run over (record, row, levels), so the launch overhead and
// the ramp-up / tail of the persistent grid are paid once per batch instead of once per record.
static int cdfmoc_gpu_compute_device_batch_dev(const float *const *d_zv, double *const *d_dmoc, int nrec, void *stream)
{
    REQUIRE_INIT();
    REQUIRE(moc.ready, CDFGPU_ERR_STATE, "cdfmoc_gpu_compute_device_batch: cdfmoc_gpu_setup has not been called");
    REQUIRE(d_zv && d_dmoc && nrec >= 1, CDFGPU_ERR_ARG, "cdfmoc_gpu_compute_device_batch: bad argument");
    {
        const double units = (double)nrec * moc.ny * (moc.nz - 1);
        REQUIRE(units < 2.0e9, CDFGPU_ERR_ARG, "cdfmoc_gpu_compute_device_batch: too many work units for one launch");
    }
    for (int r = 0; r < nrec; ++r) REQUIRE(d_zv[r] && d_dmoc[r], CDFGPU_ERR_ARG, "cdfmoc_gpu_compute_device_batch: null pointer");
    cudaStream_t st = stream ? (cudaStream_t)stream : g.s_compute;
    if (nrec == 1) return cdfmoc_gpu_compute_device_dev(d_zv[0], d_dmoc[0], stream);
    if (nrec > moc.batch_cap) {
        CDF_CUDA(cudaDeviceSynchronize());   // (re)allocation of the pointer tables: rare, and no launch may still read them
        cudaFree(moc.d_batch_zv); cudaFree(moc.d_batch_out); cudaFree(moc.d_batch_col);
        moc.d_batch_zv = nullptr; moc.d_batch_out = nullptr; moc.d_batch_col = nullptr;
        moc.batch_cap = 0;
        CDF_CUDA(cudaMalloc(&moc.d_batch_zv, (size_t)2 * nrec * sizeof(float *)));    // two tables in rotation: the copy for launch
        CDF_CUDA(cudaMalloc(&moc.d_batch_out, (size_t)2 * nrec * sizeof(double *)));  // N+1 must not overwrite launch N's
        CDF_CUDA(cudaMalloc(&moc.d_batch_col, (size_t)nrec * moc.ny * sizeof(int)));
        CDF_CUDA(cudaMemsetAsync(moc.d_batch_col, 0, (size_t)nrec * moc.ny * sizeof(int), st));
        moc.batch_cap = nrec;
        moc.batch_flip = 0;
    }
    // stream-ordered copies of the pointer tables (pageable source: the runtime stages them before returning)
    const float **tz = moc.d_batch_zv + (size_t)moc.batch_flip * moc.batch_cap;
    double **to = moc.d_batch_out + (size_t)moc.batch_flip * moc.batch_cap;
    moc.batch_flip ^= 1;
    CDF_CUDA(cudaMemcpyAsync(tz, d_zv, (size_t)nrec * sizeof(float *), cudaMemcpyHostToDevice, st));
    CDF_CUDA(cudaMemcpyAsync(to, d_dmoc, (size_t)nrec * sizeof(double *), cudaMemcpyHostToDevice, st));
    // the pointer tables are written on this stream right before the kernel: no load ahead of the predecessor
    return moc_launch(d_zv[0], d_dmoc[0], stream ? moc.ws_ext : moc.ws_int, st, 0, true, nrec, tz, to, moc.d_batch_col);
}

static int cdfmoc_gpu_maxmoc_dev(int slot, int basin, int ijmin, int ijmax, int ikmin, int ikmax, float *ovt, int *loc)
{
    REQUIRE_INIT();
    REQUIRE(moc.ready, CDFGPU_ERR_STATE, "cdfmoc_gpu_maxmoc: cdfmoc_gpu_setup has not been called");
    REQUIRE(slot >= 0 && slot < g.nslots && ovt && loc, CDFGPU_ERR_ARG, "cdfmoc_gpu_maxmoc: bad argument");
    REQUIRE(basin >= 0 && basin < moc.nb, CDFGPU_ERR_ARG, "cdfmoc_gpu_maxmoc: basin out of range");
    REQUIRE(ijmin >= 1 && ijmax <= moc.ny && ijmin <= ijmax && ikmin >= 1 && ikmax <= moc.nz && ikmin <= ikmax,
            CDFGPU_ERR_ARG, "cdfmoc_gpu_maxmoc: empty or out-of-range window");
    Slot &s = moc.slots[slot];
    REQUIRE(s.used, CDFGPU_ERR_STATE, "cdfmoc_gpu_maxmoc: nothing was submitted on this slot");
    if (!moc.d_ext) CDF_CUDA(cudaMalloc(&moc.d_ext, 4 * sizeof(float)));
    CDF_CUDA(cudaStreamWaitEvent(g.s_d2h, s.ev_k1, 0));
    const int nj = ijmax - ijmin + 1, nk = ikmax - ikmin + 1;
    moc_window_extrema_kernel<<<1, 256, 0, g.s_d2h>>>(s.d_out, moc.ny, moc.nb, basin, ijmin - 1, nj, ikmin - 1, nk,
                                                     moc.d_ext, reinterpret_cast<int *>(moc.d_ext + 2));
    CDF_CUDA(cudaGetLastError());
    ++g.launches;
    float h[4];
    CDF_CUDA(cudaMemcpyAsync(h, moc.d_ext, sizeof(h), cudaMemcpyDeviceToHost, g.s_d2h));
    CDF_CUDA(cudaStreamSynchronize(g.s_d2h));
    int il[2];
    memcpy(il, h + 2, sizeof(il));
    ovt[0] = h[0]; ovt[1] = h[1];
    loc[0] = il[0] % nj + ijmin; loc[1] = il[0] / nj + ikmin;
    loc[2] = il[1] % nj + ijmin; loc[3] = il[1] / nj + ikmin;
    return CDFGPU_OK;
}

static int cdfmoc_gpu_decomp_setup_dev(int teos10, const float *e1u, const float *gphiv, const float *gdept, const int16_t *umask,
                            const int16_t *tmask)
{
    REQUIRE_INIT();
    REQUIRE(moc.ready, CDFGPU_ERR_STATE, "cdfmoc_gpu_decomp_setup: cdfmoc_gpu_setup has not been called");
    REQUIRE(e1u && gphiv && gdept && umask && tmask, CDFGPU_ERR_ARG, "cdfmoc_gpu_decomp_setup: null pointer");
    const size_t nxy = (size_t)moc.nx * moc.ny, n3 = nxy * (size_t)(moc.nz - 1), nout = moc.out_elems();
    // f at the V point and -g/rau0/f (cdfmoc.f90:425-433), REAL(4), with libm's sinf like the Fortran run-time
    std::vector<float> zcoef(nxy);
    {
        const float rau0 = 1025.0f, grav = 9.81f;
        const float rpi = acosf(-1.f);
        for (size_t c = 0; c < nxy; ++c) {
            volatile float f = 2 * 2 * rpi;
            f = f / (24.0f * 3600.f);
            volatile float a = rpi * gphiv[c];
            a = a / 180.0f;
            f = f * sinf(a);
            if (f != 0.f) { volatile float gg = -grav / rau0; zcoef[c] = gg / f; } else zcoef[c] = 0.f;
        }
    }
    // reference profile at every level's depth (eos.f90:843-845), plain double arithmetic on the host
    moc.dec_dlh.resize(moc.nz); moc.dec_dlref.resize(moc.nz);
    for (int k = 0; k < moc.nz; ++k) {
        const double *R = CDF_EOS_R0;
        volatile double h = (double)gdept[k] * 1.e-4;
        volatile double a = R[5] * h;
        a = a + R[4]; a = a * h; a = a + R[3]; a = a * h; a = a + R[2]; a = a * h; a = a + R[1]; a = a * h;
        a = a + R[0]; a = a * h;
        moc.dec_dlh[k] = h; moc.dec_dlref[k] = a;
    }
    moc.dec_teos10 = teos10 ? 1 : 0;
#define DALLOC(p, n) if (!(p)) CDF_CUDA(cudaMalloc(&(p), (n)))
    DALLOC(moc.d_e1u, nxy * 4); DALLOC(moc.d_zcoef, nxy * 4); DALLOC(moc.d_zt, n3 * 4); DALLOC(moc.d_zs, n3 * 4);
    DALLOC(moc.d_sig, nxy * 4); DALLOC(moc.d_hdep, nxy * 4); DALLOC(moc.d_zvgeo, n3 * 4 + 16);
    DALLOC(moc.d_umask, n3 * 2); DALLOC(moc.d_tmask, n3 * 2); DALLOC(moc.d_dvbt, nxy * 8); DALLOC(moc.d_dvgeo, 2 * nxy * 8);
    DALLOC(moc.d_sh, nout * 8); DALLOC(moc.d_bt, nout * 8); DALLOC(moc.d_ag, nout * 8); DALLOC(moc.d_btw, nout * 8);
#undef DALLOC
    CDF_CUDA(cudaMemcpyAsync(moc.d_e1u, e1u, nxy * 4, cudaMemcpyHostToDevice, g.s_compute));
    CDF_CUDA(cudaMemcpyAsync(moc.d_zcoef, zcoef.data(), nxy * 4, cudaMemcpyHostToDevice, g.s_compute));
    CDF_CUDA(cudaMemcpyAsync(moc.d_umask, umask, n3 * 2, cudaMemcpyHostToDevice, g.s_compute));
    CDF_CUDA(cudaMemcpyAsync(moc.d_tmask, tmask, n3 * 2, cudaMemcpyHostToDevice, g.s_compute));
    CDF_CUDA(cudaStreamSynchronize(g.s_compute));
    moc.decomp = true;
    return CDFGPU_OK;
}

static int cdfmoc_gpu_decomp_submit_dev(int slot, int jt, const float *zv, const float *zt, const float *zs)
{
    REQUIRE_INIT();
    REQUIRE(moc.ready && moc.decomp, CDFGPU_ERR_STATE, "cdfmoc_gpu_decomp_submit: cdfmoc_gpu_decomp_setup has not been called");
    REQUIRE(zt && zs, CDFGPU_ERR_ARG, "cdfmoc_gpu_decomp_submit: null pointer");
    // The component slabs (sh, bt, ag) and the working fields of the decomposition are plan-wide, not per slot: one
    // decomposition is in flight per device at a time -- a second submit before the fetch would overwrite the first's results
    REQUIRE(moc.dec_pending < 0 || moc.dec_pending == slot, CDFGPU_ERR_STATE,
            "cdfmoc_gpu_decomp_submit: another slot's decomposition has not been fetched yet (one record in flight per device)");
    int rc = cdfmoc_gpu_submit_dev(slot, jt, zv);   // total MOC (cdfmoc.f90:352-388) into the slot's slab
    if (rc) return rc;
    rc = ensure_eos(moc.dec_teos10, g.s_compute);
    if (rc) return rc;
    cudaStream_t st = g.s_compute;
    Slot &s = moc.slots[slot];
    const int nx = moc.nx, ny = moc.ny, nz = moc.nz, nzm1 = nz - 1;
    const size_t nxy = (size_t)nx * ny, nout = moc.out_elems();
    const int gsz = g.sm_count * 8;
    // T and S go to the plan-wide fields on the compute stream (packed ones through the slot's staging buffers)
    if ((rc = field_h2d_in(kCallSubmit, 1, moc.d_zt, s.d_stage[1], zt, (size_t)nzm1, nxy, st)) ||
        (rc = field_h2d_in(kCallSubmit, 2, moc.d_zs, s.d_stage[2], zs, (size_t)nzm1, nxy, st)))
        return rc;
    // 2.1 barotropic: vertical mean of V, weighted zonal sums, integration (:397-419)
    decomp_vbar_kernel<<<gsz, 256, 0, st>>>(moc.d_e3m, s.d_in[0], nxy, nzm1, 0, moc.d_hdep, 1, moc.d_dvbt);
    if ((rc = decomp_weighted(moc.d_dvbt, moc.d_bt, st))) return rc;
    decomp_scan_kernel<<<(ny * moc.nb + 127) / 128, 128, 0, st>>>(moc.d_bt, nullptr, ny * moc.nb, nz);
    // 2.2 geostrophic shear: level by level from the bottom (:435-478)
    CDF_CUDA(cudaMemsetAsync(moc.d_dvgeo, 0, 2 * nxy * 8, st));
    int iup = 0, ido = 1;
    for (int k = nzm1 - 1; k >= 0; --k) {
        decomp_sigma_kernel<<<gsz, 256, 0, st>>>(moc.d_zt + (size_t)k * nxy, moc.d_zs + (size_t)k * nxy,
                                                 moc.d_tmask + (size_t)k * nxy, moc.dec_dlh[k], moc.dec_dlref[k], nxy, moc.d_sig);
        decomp_geo_level_kernel<<<gsz, 256, 0, st>>>(moc.d_sig, moc.d_umask + (size_t)k * nxy, moc.d_e1u, moc.d_zcoef,
                                                     moc.d_ibmask, moc.nb, moc.d_e3m + (size_t)k * nxy,
                                                     s.d_in[0] + (size_t)(nzm1 - 1) * nxy, moc.d_dvgeo + (size_t)ido * nxy,
                                                     moc.d_dvgeo + (size_t)iup * nxy, moc.d_zvgeo + (size_t)k * nxy, nx, ny);
        std::swap(iup, ido);
        g.launches += 2;
    }
    CDF_CUDA(cudaGetLastError());
    // zonal sums of the geostrophic velocity (K1 without its scan), its pseudo-barotropic part, integration (:464-510)
    if ((rc = moc_launch(moc.d_zvgeo, moc.d_sh, moc.ws_int, st, 1))) return rc;
    decomp_vbar_kernel<<<gsz, 256, 0, st>>>(moc.d_e3m, moc.d_zvgeo, nxy, nzm1, 1, moc.d_hdep, 0, moc.d_dvbt);
    if ((rc = decomp_weighted(moc.d_dvbt, moc.d_btw, st))) return rc;
    decomp_scan_kernel<<<(ny * moc.nb + 127) / 128, 128, 0, st>>>(moc.d_sh, moc.d_btw, ny * moc.nb, nz);
    // 2.3 ageostrophic (:516)
    decomp_ageo_kernel<<<gsz, 256, 0, st>>>(s.d_out, moc.d_sh, moc.d_bt, moc.d_ag, nout);
    CDF_CUDA(cudaGetLastError());
    g.launches += 5;
    CDF_CUDA(cudaEventRecord(s.ev_k1, st));
    moc.dec_pending = slot;
    return CDFGPU_OK;
}

static int cdfmoc_gpu_decomp_fetch_dev(int slot, double *dmoc, double *dmoc_sh, double *dmoc_bt, double *dmoc_ag)
{
    REQUIRE_INIT();
    REQUIRE(moc.ready && moc.decomp, CDFGPU_ERR_STATE, "cdfmoc_gpu_decomp_fetch: cdfmoc_gpu_decomp_setup has not been called");
    REQUIRE(dmoc && dmoc_sh && dmoc_bt && dmoc_ag, CDFGPU_ERR_ARG, "cdfmoc_gpu_decomp_fetch: null pointer");
    REQUIRE(moc.dec_pending == slot, CDFGPU_ERR_STATE,
            "cdfmoc_gpu_decomp_fetch: this slot holds no pending decomposition (the components belong to the latest decomp_submit)");
    int rc = cdfmoc_gpu_fetch_dev(slot, dmoc);
    if (rc) return rc;
    const size_t nb8 = moc.out_elems() * sizeof(double);
    CDF_CUDA(cudaMemcpyAsync(dmoc_sh, moc.d_sh, nb8, cudaMemcpyDeviceToHost, g.s_d2h));
    CDF_CUDA(cudaMemcpyAsync(dmoc_bt, moc.d_bt, nb8, cudaMemcpyDeviceToHost, g.s_d2h));
    CDF_CUDA(cudaMemcpyAsync(dmoc_ag, moc.d_ag, nb8, cudaMemcpyDeviceToHost, g.s_d2h));
    CDF_CUDA(cudaStreamSynchronize(g.s_d2h));
    moc.dec_pending = -1;
    return CDFGPU_OK;
}

static int cdfmoc_gpu_kernel_ms_dev(int slot, float *ms)
{
    REQUIRE_INIT();
    REQUIRE(moc.ready && slot >= 0 && slot < g.nslots && ms, CDFGPU_ERR_ARG, "cdfmoc_gpu_kernel_ms: bad argument");
    Slot &s = moc.slots[slot];
    REQUIRE(s.used, CDFGPU_ERR_STATE, "cdfmoc_gpu_kernel_ms: nothing was submitted on this slot");
    CDF_CUDA(cudaEventSynchronize(s.ev_k1));
    CDF_CUDA(cudaEventElapsedTime(ms, s.ev_k0, s.ev_k1));
    return CDFGPU_OK;
}

}  // extern "C"

#include "api_mocsig.inc"
#include "api_zonal.inc"
#include "api_transig.inc"
#include "api_sigtrp.inc"
#include "api_multi.inc"
