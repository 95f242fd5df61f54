// host_common.hpp -- shared host logic of the C++ twins of cdfmoc / cdfmocsig (names, files, masks, output file).
// Mirrors, for the hot path only: src/modcdfnames.F90:17-187,362-388 (default names, CDFT_* environment),
// src/cdfio.F90 (chkfile :3032-3070, SetMeshZgrVersion :3310-3335, getvar name mapping :1510-1536, getvare3 :2221-2274),
// src/cdfmoc.f90:325-336 / src/cdfmocsig.f90:347-359 (basin mask assembly), cdfmoc.f90:1019-1028,1182-1186 (output).
#pragma once
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>

#include <ctype.h>

#include <chrono>
#include <fstream>
#include <map>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/cdfgpu.h"
#include "nc3.hpp"

namespace cdfhost {

struct Names {  // modcdfnames.F90 defaults
    std::string x = "x", y = "y", z = "depth", t = "time_counter";
    std::string vomecrty = "vomecrty", vomeeivv = "vomeeivv", votemper = "votemper", vosaline = "vosaline";
    std::string e1v = "e1v", e1u = "e1u", gphiv = "gphiv", vmask = "vmask", umask = "umask", tmask = "tmask", tmaskatl = "tmaskatl",
                tmaskind = "tmaskind", tmaskpac = "tmaskpac", vtimec = "time_counter", vdepthw = "depthw", vlon2d = "nav_lon",
                vlat2d = "nav_lat", ve3v = "e3v", ve3vvvl = "e3v", ve3t1d = "e3t", gdept = "gdept", gdepw = "gdepw";
    std::string fhgr = "mesh_hgr.nc", fzgr = "mesh_zgr.nc", fmsk = "mask.nc", fbasins = "new_maskglo.nc";
    std::string missing = "_FillValue";
    Names()
    {
        read_cdf_names();
        chkenv();
    }
    void chkenv()
    {  // modcdfnames.F90:376-380
        auto env = [](const char *n, std::string &dst) { const char *e = getenv(n); if (e && *e) dst = e; };
        env("CDFT_MESH_HGR", fhgr); env("CDFT_MESH_ZGR", fzgr); env("CDFT_MASK", fmsk); env("CDFT_BASINS", fbasins);
    }
    // ReadCdfNames (modcdfnames.F90:268-326): the namelist nam_cdf_names ($NAM_CDF_NAMES) in the current directory, else in
    // $HOME/CDFTOOLS_cfg/, renames dimensions, variables and mesh / mask files.  The reference READs the groups namdim,
    // namdimvar, nammetrics, namvars, nambathy, namsqdvar and nammeshmask (NOT nammask: the mask variable names cannot be
    // changed this way there either); unknown keys are ignored here where the Fortran run-time would stop.
    void read_cdf_names()
    {
        std::string nam = "nam_cdf_names";
        if (const char *e = getenv("NAM_CDF_NAMES")) if (*e) nam = e;
        struct stat st;
        if (stat(nam.c_str(), &st) != 0) {
            const char *home = getenv("HOME");
            nam = std::string(home ? home : "") + "/CDFTOOLS_cfg/" + nam;
            if (stat(nam.c_str(), &st) != 0) return;
        }
        printf("  CAUTION : dim names and variable names are now set according to \n  =======   the following namelist : %s\n", nam.c_str());
        std::ifstream f(nam);
        std::stringstream ss;
        ss << f.rdbuf();
        const std::map<std::string, std::map<std::string, std::string *>> groups = {
            {"namdim", {{"cn_x", &x}, {"cn_y", &y}, {"cn_z", &z}, {"cn_t", &t}}},
            {"namdimvar", {{"cn_vlon2d", &vlon2d}, {"cn_vlat2d", &vlat2d}, {"cn_vdepthw", &vdepthw}, {"cn_vtimec", &vtimec},
                           {"cn_missing_value", &missing}}},
            {"nammetrics", {{"cn_ve1v", &e1v}, {"cn_ve1u", &e1u}, {"cn_gphiv", &gphiv}, {"cn_ve3v", &ve3v}, {"cn_ve3vvvl", &ve3vvvl},
                            {"cn_ve3t1d", &ve3t1d}, {"cn_gdept", &gdept}, {"cn_gdepw", &gdepw}}},
            {"namvars", {{"cn_vomecrty", &vomecrty}, {"cn_vomeeivv", &vomeeivv}, {"cn_votemper", &votemper}, {"cn_vosaline", &vosaline}}},
            {"nammeshmask", {{"cn_fzgr", &fzgr}, {"cn_fhgr", &fhgr}, {"cn_fmsk", &fmsk}, {"cn_fbasins", &fbasins}}},
        };
        parse_namelist(ss.str(), groups);
    }
    // a Fortran namelist file, as far as character assignments go:  &group  key = 'value' [,] ...  /   ; ! starts a comment
    static void parse_namelist(const std::string &txt, const std::map<std::string, std::map<std::string, std::string *>> &groups)
    {
        auto lower = [](std::string v) { for (auto &c : v) c = (char)tolower((unsigned char)c); return v; };
        std::string clean;   // comments out (outside quotes)
        {
            char q = 0;
            bool com = false;
            for (char c : txt) {
                if (com) { if (c == '\n') { com = false; clean += c; } continue; }
                if (q) { if (c == q) q = 0; clean += c; continue; }
                if (c == '\'' || c == '"') { q = c; clean += c; continue; }
                if (c == '!') { com = true; continue; }
                clean += c;
            }
        }
        size_t pos = 0;
        while ((pos = clean.find('&', pos)) != std::string::npos) {
            size_t e = pos + 1;
            while (e < clean.size() && (isalnum((unsigned char)clean[e]) || clean[e] == '_')) ++e;
            const std::string gname = lower(clean.substr(pos + 1, e - pos - 1));
            // the group ends at the first '/' outside quotes (or at "&end")
            size_t end = e;
            char q = 0;
            for (; end < clean.size(); ++end) {
                const char c = clean[end];
                if (q) { if (c == q) q = 0; continue; }
                if (c == '\'' || c == '"') { q = c; continue; }
                if (c == '/' || c == '&') break;
            }
            const std::string body = clean.substr(e, end - e);
            pos = end + 1;
            const auto git = groups.find(gname);
            if (git == groups.end()) continue;
            size_t p2 = 0;
            while (p2 < body.size()) {
                const size_t eq = body.find('=', p2);
                if (eq == std::string::npos) break;
                size_t k1 = eq;
                while (k1 > p2 && isspace((unsigned char)body[k1 - 1])) --k1;
                size_t k0 = k1;
                while (k0 > p2 && (isalnum((unsigned char)body[k0 - 1]) || body[k0 - 1] == '_')) --k0;
                const std::string key = lower(body.substr(k0, k1 - k0));
                size_t v0 = eq + 1;
                while (v0 < body.size() && isspace((unsigned char)body[v0])) ++v0;
                std::string val;
                size_t v1 = v0;
                if (v0 < body.size() && (body[v0] == '\'' || body[v0] == '"')) {
                    const char qq = body[v0];
                    v1 = body.find(qq, v0 + 1);
                    if (v1 == std::string::npos) break;
                    val = body.substr(v0 + 1, v1 - v0 - 1);
                    ++v1;
                } else {
                    while (v1 < body.size() && !isspace((unsigned char)body[v1]) && body[v1] != ',') ++v1;
                    val = body.substr(v0, v1 - v0);
                }
                while (!val.empty() && val.back() == ' ') val.pop_back();   // CHARACTER(LEN=256) values are used TRIMmed
                const auto kit = git->second.find(key);
                if (kit != git->second.end()) *kit->second = val;
                p2 = v1;
            }
        }
    }
};

// $CDFGPU_TIMING=1: wall-clock seconds of the phases of a run on stderr ("<tool>: phase <name> <seconds>")
struct PhaseTimer {
    const char *tool;
    bool on;
    std::chrono::steady_clock::time_point t0, last;
    explicit PhaseTimer(const char *t) : tool(t), on(getenv("CDFGPU_TIMING") && atoi(getenv("CDFGPU_TIMING")))
    {
        t0 = last = std::chrono::steady_clock::now();
    }
    void mark(const char *name)
    {
        const auto now = std::chrono::steady_clock::now();
        if (on) fprintf(stderr, "%s: phase %s %.3f\n", tool, name, std::chrono::duration<double>(now - last).count());
        last = now;
    }
    void total()
    {
        if (on) fprintf(stderr, "%s: phase total %.3f\n", tool, std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
    }
};

// CUDA context creation overlaps the reading of the mesh / mask files: a helper thread creates the contexts while the
// main thread reads; join() before cdfgpu_init
struct CudaWarmup {
    std::thread th;
    CudaWarmup() : th([] { cdfgpu_warmup(); }) {}
    void join() { if (th.joinable()) th.join(); }
    ~CudaWarmup() { join(); }
};

// -nc4: the reference builds without key_netcdf4 accept the flag and write 64-bit-offset classic files all the same
// (src/cdfio.F90:291-299: NF90_NETCDF4 only under the CPP key); so does this twin, and says so once
inline void note_nc4()
{
    printf("  -nc4 : this build has no NetCDF-4 / HDF5 writer; output is 64-bit offset classic NetCDF, as from a\n"
           "         reference build without key_netcdf4 (cdfio.F90:291-299)\n");
}

// chkfile (cdfio.F90:3032-3070): returns true when the file is MISSING (and says so), like the reference
inline bool chkfile(const std::string &f, bool verbose = true)
{
    if (f == "none") return false;
    struct stat st;
    if (stat(f.c_str(), &st) == 0) return false;
    if (verbose) printf(" %s is missing \n", f.c_str());
    return true;
}

[[noreturn]] inline void stop(int code) { fflush(stdout); exit(code); }
inline void gpu_check(int rc, const char *where)
{
    if (rc == CDFGPU_OK) return;
    printf(" ERROR in %s : libcdfgpu status %d : %s\n", where, rc, cdfgpu_last_error());
    stop(97);
}
inline void nc_check(bool ok, const std::string &err)
{
    if (ok) return;
    printf(" ERROR : %s\n", err.c_str());
    stop(98);  // the reference STOPs 98 on NetCDF errors (cdfio.F90:2937)
}

struct MeshZgr {
    nc3::Reader nc;
    std::string ver;   // v2.0 | v3.0 | v3.6  (SetMeshZgrVersion, cdfio.F90:3310-3335)
    void open(const std::string &path)
    {
        nc_check(nc.open(path), nc.err);
        const int iv = nc.find_var("e3t_0");
        if (iv < 0) ver = "v2.0";   // IOIPSL-style file: e3._ps, gdept / gdepw / e3t as (t,z,1,1) columns
        else {
            int nsp = 0;  // number of non-record, non-singleton dims
            for (int d : nc.vars[iv].dimids) if (nc.dims[d].len > 1 && d != nc.recdim) ++nsp;
            ver = (nsp <= 1) ? "v3.0" : "v3.6";
        }
        printf("  mesh_zgr version is %s\n", ver.c_str());
    }
    // getvar(..., ldiom=.true.) maps cn_ve3v (cdfio.F90:1522-1527)
    std::string e3v_name(const std::string &cn_ve3v = "e3v") const
    {
        (void)cn_ve3v;
        return ver == "v2.0" ? "e3v_ps" : ver == "v3.0" ? "e3v" : "e3v_0";
    }
    std::string name1d(const std::string &base) const  // getvare3 (cdfio.F90:2232-2274): gdepw / gdept / e3t1d
    {
        if (base == "gdepw") return ver == "v2.0" ? "gdepw" : ver == "v3.0" ? "gdepw_0" : "gdepw_1d";
        if (base == "gdept") return ver == "v2.0" ? "gdept" : ver == "v3.0" ? "gdept_0" : "gdept_1d";
        return ver == "v2.0" ? "e3t" : ver == "v3.0" ? "e3t_0" : "e3t_1d";
    }
};

// the variable `var` of `nc`; STOP 98 when the file has none, as getvar does on a NetCDF error
inline const nc3::Var &var_or_die(nc3::Reader &nc, const std::string &var)
{
    const int iv = nc.find_var(var);
    if (iv < 0) { printf(" ERROR : variable %s not found in %s\n", var.c_str(), nc.path.c_str()); stop(98); }
    return nc.vars[iv];
}

// one (ny,nx) level of a (t,z,y,x) / (z,y,x) / (y,x) variable, like getvar(cdfile, cdvar, klev, kpi, kpj, ktime)
inline void read_level(nc3::Reader &nc, const std::string &var, int klev /*0-based*/, long rec, size_t nxy, float *out)
{
    const nc3::Var &v = var_or_die(nc, var);
    const uint64_t nlev = v.nelem_per_rec / nxy;
    const uint64_t off = (nlev > 1 ? (uint64_t)klev : 0) * nxy;
    nc_check(nc.read_f32(v, v.isrec ? rec : 0, off, nxy, out), nc.err);
}
inline void read_1d(nc3::Reader &nc, const std::string &var, size_t n, float *out)
{
    nc_check(nc.read_f32(var_or_die(nc, var), 0, 0, n, out), nc.err);
}

// ibmask(nb,nx,ny): 1 global(vmask k=1), 2 atl, 3 indo-pacific = min(1,pac+ind), 4 ind, 5 pac  (cdfmoc.f90:325-336)
inline void basin_masks(const Names &cn, bool lbas, int nx, int ny, bool zero_edges, std::vector<int16_t> &ib)
{
    const int nb = lbas ? 5 : 1;
    const size_t nxy = (size_t)nx * ny;
    ib.assign(nxy * nb, 0);
    std::vector<float> tmp(nxy);
    nc3::Reader msk;
    nc_check(msk.open(cn.fmsk), msk.err);
    read_level(msk, cn.vmask, 0, 0, nxy, tmp.data());
    for (size_t c = 0; c < nxy; ++c) ib[c * nb] = (int16_t)tmp[c];
    if (lbas) {
        nc3::Reader bas;
        nc_check(bas.open(cn.fbasins), bas.err);
        const std::string *names[3] = {&cn.tmaskatl, &cn.tmaskind, &cn.tmaskpac};
        const int slot[3] = {1, 3, 4};
        for (int m = 0; m < 3; ++m) {
            read_level(bas, *names[m], 0, 0, nxy, tmp.data());
            for (size_t c = 0; c < nxy; ++c) ib[c * nb + slot[m]] = (int16_t)tmp[c];
        }
        for (size_t c = 0; c < nxy; ++c) {
            int16_t s = (int16_t)(ib[c * nb + 4] + ib[c * nb + 3]);
            ib[c * nb + 2] = s > 0 ? (int16_t)1 : s;
        }
    }
    if (zero_edges)
        for (int j = 0; j < ny; ++j) { ib[((size_t)j * nx) * nb] = 0; ib[((size_t)j * nx + nx - 1) * nb] = 0; }
}

// nav_lat(1,:) = gphiv(iloc(1),:) with iloc = MAXLOC(gphiv) (cdfmoc.f90:316-318): first maximum in column-major order
inline void dummy_lat(const std::vector<float> &gphiv, int nx, int ny, std::vector<float> &lat)
{
    size_t imax = 0;
    float best = gphiv[0];
    for (size_t c = 1; c < (size_t)nx * ny; ++c)
        if (gphiv[c] > best) { best = gphiv[c]; imax = c; }
    const int i = (int)(imax % nx);
    lat.resize(ny);
    for (int j = 0; j < ny; ++j) lat[j] = gphiv[(size_t)j * nx + i];
}

struct OutVar { std::string name, long_name, units; float valid_min, valid_max; float fill = 99999.f; std::string axis = "TZY"; std::string short_name = ""; };

// create + createvar + putheadervar + putvar1d for the (t, depth|sigma, y, x=1) output files
// (cdfio.F90:260-368,371-459,629-682,2290-2407; cdfmoc.f90:1019-1028,1182-1186; cdfmocsig.f90:502-510,576-581)
struct OutFile {
    nc3::Writer w;
    std::vector<int> varids;
    int ny = 0, nlev = 0;
    void create(const std::string &path, const std::string &zdim, int ny_, int nlev_, const std::vector<OutVar> &vars,
                const std::string &history, const std::vector<float> &navlat, const std::vector<float> &zaxis,
                const std::vector<double> &tim, nc3::Reader &ref)
    {
        ny = ny_; nlev = nlev_;
        const int dx = w.def_dim("x", 1), dy = w.def_dim("y", ny), dz = w.def_dim(zdim, nlev), dt = w.def_dim("time_counter", 0);
        const int vlon = w.def_var("nav_lon", nc3::NC_FLOAT, {dy, dx});
        const int vlat = w.def_var("nav_lat", nc3::NC_FLOAT, {dy, dx});
        const int vz = w.def_var(zdim, nc3::NC_FLOAT, {dz});
        const int vt = w.def_var("time_counter", nc3::NC_DOUBLE, {dt});
        // copyatt of the time variable from the reference file (cdfio.F90:353-354)
        const int it = ref.find_var("time_counter");
        if (it >= 0)
            for (auto &a : ref.vars[it].atts)
                if (a.type == nc3::NC_CHAR) w.put_att_text(vt, a.name, a.as_string());
        // global attributes (cdfio.F90:360-363) taken from the reference file when present (getdim caches them, :939-994)
        auto gatt = [&](const char *n, const char *dflt) {
            for (auto &a : ref.gatts) if (a.name == n && a.type == nc3::NC_CHAR) return a.as_string();
            return std::string(dflt);
        };
        int start_date = -1;
        for (auto &a : ref.gatts) if (a.name == "start_date") start_date = (int)a.as_double();
        w.put_att_int(-1, "start_date", start_date);
        w.put_att_text(-1, "output_frequency", gatt("output_frequency", "N/A"));
        w.put_att_text(-1, "CONFIG", gatt("CONFIG", "N/A"));
        w.put_att_text(-1, "CASE", gatt("CASE", "N/A"));
        for (auto &v : vars) {
            const int id = w.def_var(v.name, nc3::NC_FLOAT, {dt, dz, dy, dx});
            w.put_att_text(id, "units", v.units);
            w.put_att_float(id, "_FillValue", v.fill);
            w.put_att_float(id, "valid_min", v.valid_min);
            w.put_att_float(id, "valid_max", v.valid_max);
            w.put_att_text(id, "long_name", v.long_name);
            w.put_att_text(id, "short_name", v.short_name.empty() ? v.name : v.short_name);
            w.put_att_int(id, "iweight", 1);
            w.put_att_text(id, "online_operation", "N/A");
            w.put_att_text(id, "axis", v.axis);
            w.put_att_float(id, "scale_factor", 1.f);
            w.put_att_float(id, "add_offset", 0.f);
            w.put_att_float(id, "savelog10", 0.f);
            varids.push_back(id);
        }
        w.put_att_text(-1, "history", history);
        nc_check(w.create(path), w.err);
        std::vector<float> zero(ny, 0.f);
        w.put_f32(vlon, 0, 0, ny, zero.data());
        w.put_f32(vlat, 0, 0, ny, navlat.data());
        w.put_f32(vz, 0, 0, nlev, zaxis.data());
        for (size_t r = 0; r < tim.size(); ++r) w.put_f64(vt, (long)r, 0, 1, &tim[r]);
    }
    // one record of one variable: vals[lev][j]
    void put(int v, long rec, const float *vals) { nc_check(w.put_f32(varids[v], rec, 0, (uint64_t)nlev * ny, vals), w.err); }
};

// ---- Fortran edit descriptors, as gfortran prints them (the ASCII outputs of the tools) --------------------------------
// Fortran E16.7: 0.ddddddd scaled, exponent of two digits
inline std::string fortran_e16_7(double x)
{
    char b[64];
    if (x == 0.0 || !std::isfinite(x)) {
        snprintf(b, sizeof b, "%16s", !std::isfinite(x) ? (std::isnan(x) ? "NaN" : (x > 0 ? "Infinity" : "-Infinity")) : "0.0000000E+00");
        return b;
    }
    snprintf(b, sizeof b, "%.6E", fabs(x));   // d.ddddddE+xx, correctly rounded to 7 significant digits
    const int ex = atoi(strchr(b, 'E') + 1) + 1;
    std::string dig;
    dig += b[0];
    dig.append(b + 2, 6);
    char o[64];
    snprintf(o, sizeof o, "%s0.%sE%c%02d", x < 0 ? "-" : "", dig.c_str(), ex < 0 ? '-' : '+', abs(ex));
    snprintf(b, sizeof b, "%16s", o);
    return b;
}

// Fortran Fw.d edit descriptor: right-justified, asterisks when the value does not fit; d = 0 keeps the decimal point
inline std::string fortran_f(double x, int w, int d)
{
    char b[64];
    if (std::isnan(x)) snprintf(b, sizeof b, "%*s", w, "NaN");
    else if (std::isinf(x)) snprintf(b, sizeof b, "%*s", w, x > 0 ? "Infinity" : "-Infinity");
    else if (d == 0) snprintf(b, sizeof b, "%*.0f.", w - 1, x);
    else snprintf(b, sizeof b, "%*.*f", w, d, x);
    std::string r = b;
    if ((int)r.size() > w) {   // gfortran drops the optional leading zero before giving up
        const size_t z = r.find("0.");
        if (z != std::string::npos && (z == 0 || r[z - 1] == '-' || r[z - 1] == ' ') && (int)r.size() == w + 1) r.erase(z, 1);
    }
    if ((int)r.size() > w) r.assign(w, '*');
    return r;
}

// End of a command-line run, after the output files are closed: the process is about to exit, so the page-locked buffers
// (cudaFreeHost of several GB costs ~0.1 s per GB) and the CUDA context are left to the operating system.  The device is
// idle at this point (every record has been fetched).  $CDFGPU_FULL_TEARDOWN=1 frees everything explicitly instead.
inline bool quick_exit_wanted()
{
    const char *e = getenv("CDFGPU_FULL_TEARDOWN");
    return !(e && atoi(e));
}
[[noreturn]] inline void quick_exit_now()
{
    fflush(stdout);
    fflush(stderr);
    _exit(0);
}

// pinned record buffers
struct Pinned {
    float *p = nullptr;
    explicit Pinned(size_t n) { p = (float *)cdfgpu_pinned_alloc(n * sizeof(float)); if (!p) { printf(" ERROR : %s\n", cdfgpu_last_error()); stop(97); } }
    ~Pinned() { cdfgpu_pinned_free(p); }
    Pinned(const Pinned &) = delete;
};

// One record array of a GPU call (`field`: its position among the call's arrays), read from variable `var` of `nc`.  The
// device can decode the raw file bytes of a plain float32 variable (K3 swap) or of a packed NC_SHORT one without savelog10
// whose constants are finite (K3b unpack); any other variable is converted on the host (read_f32).  Once the field is
// declared to the library, read() fills a buffer of n values the way the declaration says: raw file bytes (n INTEGER(2)
// when packed), or host-order REAL(4).
struct RecordField {
    int field;
    nc3::Reader *nc;
    const nc3::Var *v;
    float sf = 1.f, ao = 0.f, sp = 0.f;
    bool packed = false;   // raw INTEGER(2) for K3b
    bool raw = false;      // raw file bytes; until declared, whether the device can decode them
    RecordField(int field_, nc3::Reader &r, const std::string &var) : field(field_), nc(&r), v(&var_or_die(r, var))
    {
        packed = r.packed_i16(*v, &sf, &ao, &sp) && std::isfinite(sf) && std::isfinite(ao);
        raw = packed || r.is_plain_f32(*v);
    }
    // a field of a sibling call is declared on its own (cdfgpu_set_sibling_input): raw whenever the device can decode it
    void declare_sibling(int call) const
    {
        gpu_check(cdfgpu_set_sibling_input(call, field, packed ? CDFGPU_INPUT_I16 : CDFGPU_INPUT_F32, raw ? 1 : 0, sf, ao, sp),
                  "cdfgpu_set_sibling_input");
    }
    void read(long rec, size_t n, float *dst) const
    {
        nc_check(raw ? nc->read_raw(*v, rec, 0, n, dst) : nc->read_f32(*v, rec, 0, n, dst), nc->err);
    }
};

// The fields of a submit call (cdfmoc_gpu_submit, cdfmoc_gpu_decomp_submit, cdfmocsig_gpu_submit) share the one process-wide
// byte order (cdfgpu_set_input_big_endian), so they are declared together: raw when the device can decode every one of them,
// all converted on the host otherwise.
inline void declare_submit(std::vector<RecordField> &fields)
{
    bool raw = true;
    for (auto &f : fields) raw = raw && f.raw;
    for (auto &f : fields) {
        f.raw = f.raw && raw;
        f.packed = f.packed && raw;
        gpu_check(cdfgpu_set_input_packing(f.field, f.packed ? CDFGPU_INPUT_I16 : CDFGPU_INPUT_F32, f.sf, f.ao, f.sp),
                  "cdfgpu_set_input_packing");
    }
    gpu_check(cdfgpu_set_input_big_endian(raw ? 1 : 0), "cdfgpu_set_input_big_endian");
}
// a field filled on the host (e3 with -vvl -full): host-order REAL(4)
inline void sibling_host_f32(int call, int field)
{
    gpu_check(cdfgpu_set_sibling_input(call, field, CDFGPU_INPUT_F32, 0, 1.f, 0.f, 0.f), "cdfgpu_set_sibling_input");
}

}  // namespace cdfhost
