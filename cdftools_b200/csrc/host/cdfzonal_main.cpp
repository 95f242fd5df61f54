// cdfzonalsum_gpu / cdfzonalmean_gpu -- C++ twins of the cdfzonalsum and cdfzonalmean command lines
// (src/cdfzonalsum.f90, src/cdfzonalmean.f90) on top of libcdfgpu's C ABI; one source, built twice (-DZONAL_MEAN).
// Same options, auxiliary files, output naming (zoi<var>_<bas> / zo<var>_<bas> [_max, _min]) and exit codes.  The level /
// basin / jj / ji loop nests (cdfzonalsum.f90:301-327, cdfzonalmean.f90:301-351) are replaced by cdfzonal_gpu_sum /
// cdfzonal_gpu_mean on whole records.
#include <memory>

#include "host_common.hpp"

using namespace cdfhost;

#ifdef ZONAL_MEAN
static const char *kTool = "cdfzonalmean_gpu";
static const char *kPrefix = "zo";
#else
static const char *kTool = "cdfzonalsum_gpu";
static const char *kPrefix = "zoi";
#endif

struct InVar { int id; std::string name, units, long_name; float spval, vmin, vmax; int ipk; };

int main(int argc, char **argv)
{
    PhaseTimer tm(kTool);
    Names cn;
    if (argc == 1) {
        printf(" usage : %s -f IN-file -p C-type [-b BASIN-file] [-l LST-var] [-pdep] %s [-o OUT-file] [-debug]\n"
               "     PURPOSE : zonal %s (along the I coordinate) of every variable of IN-file, per sub-basin, on a B200 GPU.\n"
               "     REQUIRED FILES : %s, %s and %s\n",
               kTool,
#ifdef ZONAL_MEAN
               "[-max] [-ndep_in]", "mean",
#else
               "[-pdeg]", "integral",
#endif
               cn.fhgr.c_str(), cn.fzgr.c_str(), cn.fmsk.c_str());
        return 0;
    }
    std::string cf_in, ctyp, cf_basins = "none", cldum;
#ifdef ZONAL_MEAN
    std::string cf_out = "zonalmean.nc";
#else
    std::string cf_out = "zonalsum.nc";
#endif
    bool lpdep = false, lpdeg = false, lmax = false, lndep_in = false, ldebug = false, lvar = false, lchk = false;
    int npbasins = 1;
    std::vector<std::string> cv_fix;
    for (int i = 1; i < argc;) {   // cdfzonalsum.f90:140-154, cdfzonalmean.f90:144-160
        const std::string a = argv[i++];
        auto next = [&]() { return std::string(i < argc ? argv[i++] : ""); };
        if (a == "-f") cf_in = next();
        else if (a == "-p") ctyp = next();
        else if (a == "-b") { cf_basins = next(); npbasins = 5; lchk = chkfile(cf_basins); }
        else if (a == "-l") {
            lvar = true;
            std::string s = next();
            size_t p0 = 0;
            for (size_t p = 0; p <= s.size(); ++p)
                if (p == s.size() || s[p] == ',') { cv_fix.push_back(s.substr(p0, p - p0)); p0 = p + 1; }
        }
        else if (a == "-pdep") lpdep = true;
        else if (a == "-o") cf_out = next();
        else if (a == "-debug") ldebug = true;
#ifdef ZONAL_MEAN
        else if (a == "-max") lmax = true;
        else if (a == "-ndep_in") lndep_in = true;
#else
        else if (a == "-pdeg") lpdeg = true;
#endif
        else { printf(" ERROR : %s : unknown option.\n", a.c_str()); stop(99); }
    }
    (void)ldebug;
    lchk = chkfile(cn.fhgr) || lchk; lchk = chkfile(cn.fzgr) || lchk; lchk = chkfile(cn.fmsk) || lchk;
    lchk = chkfile(cf_in.empty() ? "(no -f file)" : cf_in) || lchk;
    if (lchk) stop(99);
    // metrics, latitude, mask and depth names of the C-grid point (cdfzonalsum.f90:171-195)
    std::string cv_e1, cv_e2, cv_phi, cv_msk, cv_depo, depi = "gdept";
    const char t = ctyp.empty() ? '?' : (char)toupper(ctyp[0]);
    switch (t) {
    case 'T': case 'S': cv_e1 = "e1t"; cv_e2 = "e2t"; cv_phi = "gphit"; cv_msk = "tmask"; cv_depo = "deptht"; break;
    case 'U': cv_e1 = "e1u"; cv_e2 = "e2u"; cv_phi = "gphiu"; cv_msk = "umask"; cv_depo = "depthu"; break;
    case 'V': cv_e1 = "e1v"; cv_e2 = "e2v"; cv_phi = "gphiv"; cv_msk = "vmask"; cv_depo = "depthv"; break;
    case 'F': cv_e1 = "e1f"; cv_e2 = "e2f"; cv_phi = "gphif"; cv_msk = "fmask"; cv_depo = "deptht"; break;
    case 'W': cv_e1 = "e1t"; cv_e2 = "e2t"; cv_phi = "gphit"; cv_msk = "tmask"; cv_depo = "depthw"; depi = "gdepw"; break;
    default: printf("  C grid:%s point not known!\n", ctyp.c_str()); stop(99);
    }

    nc3::Reader in;
    nc_check(in.open(cf_in), in.err);
    const int nx = (int)in.dim_len(cn.x, true), ny = (int)in.dim_len(cn.y, false);
    int npk = (int)in.dim_len(cn.z, false);
    const int npt = (int)in.dim_len(cn.t, false);
    printf("npiglo = %d\nnpjglo = %d\nnpk    = %d\nnpt    = %d\n", nx, ny, npk, npt);
    bool l2d = false;
    if (npk <= 0) { npk = 1; l2d = true; printf(" It is a 2D field, assume npk=1 and gdep=0\n"); }
    const size_t nxy = (size_t)nx * ny;

    // input variables: 4 dims -> npk levels, 3 dims -> 1 level, else skipped (getipk, cdfio.F90:1181-1190); -l keeps the listed ones
    std::vector<InVar> vars;
    for (int iv = 0; iv < (int)in.vars.size(); ++iv) {
        const nc3::Var &v = in.vars[iv];
        const int nd = (int)v.dimids.size();
        int ipk = nd == 4 ? npk : (nd == 3 ? 1 : 0);
        if (lvar && std::find(cv_fix.begin(), cv_fix.end(), v.name) == cv_fix.end()) ipk = 0;
        if (ipk == 0) continue;
        InVar x;
        x.id = iv; x.name = v.name; x.ipk = ipk;
        const nc3::Att *a;
        x.units = (a = v.att("units")) && a->type == nc3::NC_CHAR ? a->as_string() : "N/A";
        x.long_name = (a = v.att("long_name")) && a->type == nc3::NC_CHAR ? a->as_string() : "N/A";
        x.spval = in.spval(v, cn.missing);
        x.vmin = (a = v.att("valid_min")) ? (float)a->as_double() : 0.f;
        x.vmax = (a = v.att("valid_max")) ? (float)a->as_double() : 0.f;
        vars.push_back(x);
    }
    if (vars.empty()) { printf(" ERROR : no variable to process in %s\n", cf_in.c_str()); stop(99); }

    nc3::Reader hgr, msk;
    nc_check(hgr.open(cn.fhgr), hgr.err);
    nc_check(msk.open(cn.fmsk), msk.err);
    MeshZgr zgr;
    zgr.open(cn.fzgr);
    std::vector<float> e1(nxy), e2(nxy), gphi(nxy), gdep(npk, 0.f), navlat, alpha;
    read_level(hgr, cv_e1, 0, 0, nxy, e1.data());
    read_level(hgr, cv_e2, 0, 0, nxy, e2.data());
    read_level(hgr, cv_phi, 0, 0, nxy, gphi.data());
    if (!l2d) read_1d(zgr.nc, zgr.name1d(depi), npk, gdep.data());
#ifdef ZONAL_MEAN
    if (lndep_in) for (auto &d : gdep) d = -1.f * d;   // cdfzonalmean.f90:272
#endif
    if (!lpdep) for (auto &d : gdep) d = -1.f * d;
    if (lpdeg) {   // alpha(:) = e2(1,:)*360./z2pi/ra, REAL(4) (cdfzonalsum.f90:260-262)
        const float z2pi = 2.0f * acosf(-1.f), ra = 6371229.f;
        alpha.resize(ny);
        for (int j = 0; j < ny; ++j) alpha[j] = ((e2[(size_t)j * nx] * 360.f) / z2pi) / ra;
    }
    dummy_lat(gphi, nx, ny, navlat);

    // basin masks (cdfzonalsum.f90:286-296): REAL(4), no zeroing of the periodic columns
    std::vector<float> zmask(nxy * npbasins, 0.f), tmp(nxy);
    read_level(msk, cv_msk, 0, 0, nxy, tmp.data());
    for (size_t c = 0; c < nxy; ++c) zmask[c * npbasins] = tmp[c];
    if (npbasins == 5) {
        nc3::Reader bas;
        nc_check(bas.open(cf_basins), bas.err);
        const std::string *names[3] = {&cn.tmaskatl, &cn.tmaskind, &cn.tmaskpac};
        const int slot[3] = {1, 3, 4};
        for (int m = 0; m < 3; ++m) {
            read_level(bas, *names[m], 0, 0, nxy, tmp.data());
            for (size_t c = 0; c < nxy; ++c) zmask[c * 5 + slot[m]] = tmp[c];
        }
        for (size_t c = 0; c < nxy; ++c) { float z = zmask[c * 5 + 4] + zmask[c * 5 + 3]; zmask[c * 5 + 2] = z > 0.f ? 1.f : z; }
    }
    std::vector<float> mvar3(nxy * (size_t)npk);
    for (int k = 0; k < npk; ++k) read_level(msk, cv_msk, k, 0, nxy, mvar3.data() + (size_t)k * nxy);

    // ---- output file (CreateOutput, cdfzonalsum.f90:369-437 / cdfzonalmean.f90:398-470)
    const char *cbasin[5] = {"_glo", "_atl", "_inp", "_ind", "_pac"};
    if (lpdeg && cf_out == "zonalsum.nc") cf_out = "zonalintdeg.nc";
    nc3::Writer w;
    const int dx = w.def_dim("x", 1), dy = w.def_dim("y", ny), dz = w.def_dim(cv_depo, npk), dt = w.def_dim("time_counter", 0);
    const int vlon = w.def_var("nav_lon", nc3::NC_FLOAT, {dy, dx}), vlat = w.def_var("nav_lat", nc3::NC_FLOAT, {dy, dx});
    const int vz = w.def_var(cv_depo, nc3::NC_FLOAT, {dz}), vt = w.def_var("time_counter", nc3::NC_DOUBLE, {dt});
    const int ncoef = lmax ? 3 : 1;
    const int nvo = (int)vars.size() * npbasins;
    std::vector<int> ids((size_t)ncoef * nvo);
    for (int q = 0; q < ncoef; ++q)
        for (size_t iv = 0; iv < vars.size(); ++iv)
            for (int b = 0; b < npbasins; ++b) {
                const InVar &x = vars[iv];
                std::string stem = x.name.size() > 2 ? x.name.substr(2) : std::string();
                const std::pair<const char *, const char *> dup[9] = {{"iowaflup", "waflio"}, {"cfc11", "cfc11"}, {"bombc14", "bc14"},
                    {"invcfc", "invcfc"}, {"invc14", "invc14"}, {"qtrcfc", "qtrcfc"}, {"qtrc14", "qtrc14"}, {"qintcfc", "qintcfc"}, {"qintc14", "qintc14"}};
                for (auto &d : dup) if (x.name == d.first) stem = d.second;
                std::string name = std::string(kPrefix) + stem + cbasin[b];
#ifdef ZONAL_MEAN
                std::string units = x.units, lname = "Zonal_Mean_" + x.long_name + cbasin[b];
                const float fill = 0.f;   // zspval (cdfzonalmean.f90:47)
                if (q == 1) { name += "_max"; lname = "Zonal_Max_" + lname.substr(11); }
                if (q == 2) { name += "_min"; lname = "Zonal_Min_" + lname.substr(11); }
#else
                std::string units = x.units + (lpdeg ? ".m2.degree-1" : ".m2");
                std::string lname = std::string(lpdeg ? "Zonal_Integral_per_degree_" : "Zonal_Integral_") + x.long_name + cbasin[b];
                const float fill = x.spval;
#endif
                const int id = x.ipk == 1 ? w.def_var(name, nc3::NC_FLOAT, {dt, dy, dx}) : w.def_var(name, nc3::NC_FLOAT, {dt, dz, dy, dx});
                w.put_att_text(id, "units", units);
                w.put_att_float(id, "_FillValue", fill);
                w.put_att_float(id, "valid_min", x.vmin);
                w.put_att_float(id, "valid_max", x.vmax);
                w.put_att_text(id, "long_name", lname);
                w.put_att_text(id, "short_name", name);
                w.put_att_text(id, "online_operation", "/N/A");
                w.put_att_text(id, "axis", x.ipk == 1 ? "TY" : "TZY");
                ids[((size_t)q * vars.size() + iv) * npbasins + b] = id;
            }
    nc_check(w.create(cf_out), w.err);
    {
        std::vector<float> zero(ny, 0.f);
        w.put_f32(vlon, 0, 0, ny, zero.data());
        w.put_f32(vlat, 0, 0, ny, navlat.data());
        w.put_f32(vz, 0, 0, npk, gdep.data());
        const int it = in.find_var(cn.vtimec);
        for (int r = 0; r < npt; ++r) { double tv = 0.0; if (it >= 0) in.read_f64(in.vars[it], r, 0, 1, &tv); w.put_f64(vt, r, 0, 1, &tv); }
    }

    // ---- GPU: variables grouped by their number of levels (one plan per group); the records of a group go through the
    // record pipeline: record n+k is read into slot (n+k) mod ns while the earlier ones are in flight, and the results are
    // written in record order.  $CDFGPU_DEVICES / $CDFGPU_SHARD=time spread the slots over several devices.
    gpu_check(cdfgpu_init(-1, 3), "cdfgpu_init");
    const int ns = cdfgpu_nslots();
    tm.mark("setup");
    for (int pass = 0; pass < 2; ++pass) {
        const int nk = pass == 0 ? npk : 1;
        if (pass == 1 && npk == 1) break;
        bool any = false;
        for (auto &x : vars) any = any || x.ipk == nk;
        if (!any) continue;
        const size_t n3 = nxy * (size_t)nk, nout = (size_t)npbasins * nk * ny;
        gpu_check(cdfzonal_gpu_setup(nx, ny, nk, npbasins, e1.data(), e2.data(), zmask.data(), mvar3.data()), "cdfzonal_gpu_setup");
        std::vector<std::unique_ptr<Pinned>> zv;   // one record buffer per slot
        for (int s = 0; s < ns; ++s) zv.emplace_back(new Pinned(n3));
        std::vector<double> dz_(nout);
        std::vector<float> fmax_(lmax ? nout : 1), fmin_(lmax ? nout : 1), plane((size_t)nk * ny);
        std::vector<std::pair<size_t, int>> recs;   // (variable, time) of the records of this group, in submission order
        auto drain = [&](size_t n) {
            const size_t iv = recs[n].first;
            const int jt = recs[n].second;
            gpu_check(cdfzonal_gpu_fetch((int)(n % ns), dz_.data(), fmax_.data(), fmin_.data()), "cdfzonal_gpu_fetch");
            for (int q = 0; q < ncoef; ++q)
                for (int b = 0; b < npbasins; ++b) {
                    for (size_t e = 0; e < (size_t)nk * ny; ++e) {
                        const size_t o = (size_t)b * nk * ny + e;
                        plane[e] = q == 0 ? (float)dz_[o] : (q == 1 ? fmax_[o] : fmin_[o]);
                    }
                    nc_check(w.put_f32(ids[((size_t)q * vars.size() + iv) * npbasins + b], jt, 0, (uint64_t)nk * ny, plane.data()), w.err);
                }
        };
        for (size_t iv = 0; iv < vars.size(); ++iv) {
            const InVar &x = vars[iv];
            if (x.ipk != nk) continue;
            const RecordField fin(0, in, x.name);
            fin.declare_sibling(CDFGPU_CALL_ZONAL);   // read at submit: the records in flight keep their own declaration
            for (int jt = 0; jt < npt; ++jt) {
                const size_t n = recs.size();
                const int slot = (int)(n % ns);
                if (n >= (size_t)ns) drain(n - ns);
                recs.emplace_back(iv, jt);
                fin.read(in.vars[x.id].isrec ? jt : 0, n3, zv[slot]->p);
#ifdef ZONAL_MEAN
                gpu_check(cdfzonal_gpu_submit_mean(slot, zv[slot]->p, 0.f, lmax ? 1 : 0), "cdfzonal_gpu_submit_mean");
#else
                gpu_check(cdfzonal_gpu_submit_sum(slot, zv[slot]->p, lpdeg ? alpha.data() : nullptr), "cdfzonal_gpu_submit_sum");
#endif
            }
        }
        for (size_t n = recs.size() > (size_t)ns ? recs.size() - ns : 0; n < recs.size(); ++n) drain(n);   // before the next setup
    }
    tm.mark("records");
    w.close();
    tm.mark("output_closed");
    gpu_check(cdfgpu_finalize(), "cdfgpu_finalize");
    tm.total();
    return 0;
}
