// cdftransig_xy3d_gpu -- C++ twin of the cdftransig_xy3d command line (src/cdftransig_xy3d.f90) on top of libcdfgpu.
// Same options (-c CONFIG-CASE -l tags... [-code code] [-S] [-depref] [-nbins] [-sigmin] [-sigzoom] [-full] [-v] [-vvl]
// [-o] [-teos10]), the same DRAKKAR file sets (CONFCASE_TAG_gridU/V/T[/S].nc, modutils.f90:85-114), mesh files, output
// variables (vouxysig, vovxysig on a sigma_N axis) and exit codes (99 usage / missing file, 98 NetCDF, 97 GPU library); -nc4 is
// accepted and writes classic NetCDF, as a reference build without key_netcdf4 does.
// The reference nests levels outside tags and frames because it reads one level at a time (:370-463); with the
// accumulators resident on the device a frame (all levels) is the unit here -- see INTEGRATION.md section 4c.  Frames go
// through the library's frame pipeline (cdftransig_gpu_submit / _wait): frame n+1 is read while frame n crosses PCIe.
#include <string.h>

#include <memory>

#include "host_common.hpp"

using namespace cdfhost;

// SetFileName (modutils.f90:85-114): CONF_TAG_gridX.nc, else CONF_TAG_grid_X.nc, else STOP 97
static std::string set_file_name(const std::string &conf, const std::string &tag, const char *grid)
{
    std::string f = conf + "_" + tag + "_grid" + grid + ".nc";
    if (!chkfile(f, false)) return f;
    f = conf + "_" + tag + "_grid_" + grid + ".nc";
    if (chkfile(f, false)) { printf(" ERROR : missing grid%s or even grid_%s file \n", grid, grid); stop(97); }
    return f;
}

int main(int argc, char **argv)
{
    PhaseTimer tm("cdftransig_xy3d_gpu");
    Names cn;
    if (argc == 1) {
        printf(" usage : cdftransig_xy3d_gpu -c CONFIG-CASE -l LST-tags [-code code ] [-S] [-depref depref ] [ -nbins nbins ]\n"
               "         [-sigmin smin s-scal] [-sigzoom sminr s-scalr ] [-full ] [-v ] [-vvl ] [-o OUT-file] [-teos10]\n"
               "     PURPOSE : time average volume transport at each grid cell in density space, on a B200 GPU.\n"
               "     AVAILABLE code : 0 | 1000 (default) | 1000-acc | 2000 | none (then -depref, -nbins, -sigmin are mandatory)\n"
               "     REQUIRED FILES : %s and %s\n"
               "     OUTPUT : uvxysig.nc (vouxysig, vovxysig in m3/s)\n",
               cn.fhgr.c_str(), cn.fzgr.c_str());
        return 0;
    }
    std::string config, cldepcode = "1000", cf_out = "uvxysig.nc", clsigma = "sigma_1";
    std::vector<std::string> tags;
    float zpref = 0.f;
    int nbins = 0, iset = 0;
    double ds1min = 0, ds1scal = 0, ds1zoom = 999., ds1scalmin = 999.;
    bool lsal = false, lfull = false, lprint = false, lvvl = false, lteos10 = false;
    for (int i = 1; i < argc;) {   // cdftransig_xy3d.f90:160-183
        const std::string a = argv[i++];
        auto next = [&]() { return std::string(i < argc ? argv[i++] : ""); };
        if (a == "-c") config = next();
        else if (a == "-l") { while (i < argc && argv[i][0] != '-') tags.push_back(argv[i++]); }   // GetTagList (:478-499)
        else if (a == "-code") cldepcode = next();
        else if (a == "-depref") { zpref = (float)atof(next().c_str()); ++iset; clsigma = "sigma_" + std::to_string((int)lroundf(zpref / 1000.f)); }
        else if (a == "-nbins") { nbins = atoi(next().c_str()); ++iset; }
        else if (a == "-sigmin") {   // the usage announces "smin s-scal"; the reference reads smin only (:171) and leaves
            ds1min = atof(next().c_str());   // ds1scal unset: a second positive number is accepted here as s-scal
            char *end = nullptr;
            if (i < argc) { const double v = strtod(argv[i], &end); if (end && *end == 0 && v > 0) { ds1scal = v; ++i; } }
        }
        else if (a == "-sigzoom") { ds1zoom = atof(next().c_str()); ++iset; ds1scalmin = atof(next().c_str()); }
        else if (a == "-S") lsal = true;
        else if (a == "-full") lfull = true;
        else if (a == "-v") lprint = true;
        else if (a == "-vvl") lvvl = true;
        else if (a == "-o") cf_out = next();
        else if (a == "-nc4") note_nc4();   // cdftransig_xy3d.f90:179
        else if (a == "-teos10") lteos10 = true;
        else { printf(" ERROR : %s : unkown option.\n", a.c_str()); stop(99); }
    }
    // pre-defined parameter sets (:188-204)
    if (cldepcode == "0") { zpref = 0.f; nbins = 101; ds1min = 23.0; ds1scal = 0.03; ds1zoom = 999.; ds1scalmin = 999.; clsigma = "sigma_0"; }
    else if (cldepcode == "1000") { zpref = 1000.f; nbins = 93; ds1min = 24.2; ds1scal = 0.10; ds1zoom = 32.3; ds1scalmin = 0.05; clsigma = "sigma_1"; }
    else if (cldepcode == "1000-acc" || cldepcode == "1000-ACC") { zpref = 1000.f; nbins = 88; ds1min = 24.5; ds1scal = 0.10; ds1zoom = 999.; ds1scalmin = 999.; clsigma = "sigma_1"; }
    else if (cldepcode == "2000") { zpref = 2000.f; nbins = 174; ds1min = 29.0; ds1scal = 0.05; ds1zoom = 999.; ds1scalmin = 999.; clsigma = "sigma_2"; }
    else if (cldepcode == "none") {
        if (iset != 3) { printf("  You must set depref, nbins, sigmin  individually\n"); stop(99); }
        if (!(ds1scal > 0)) { printf(" ERROR : with -code none give the bin width too : -sigmin smin s-scal\n"); stop(99); }
    } else { printf("  This depcode :%s is not available.\n", cldepcode.c_str()); stop(99); }
    if (config.empty() || tags.empty()) { printf(" ERROR : -c CONFIG-CASE and -l LST-tags are mandatory.\n"); stop(99); }
    bool lchk = chkfile(cn.fzgr);
    lchk = chkfile(cn.fhgr) || lchk;
    if (lchk) stop(99);
    ds1scalmin = ds1scalmin < ds1scal ? ds1scalmin : ds1scal;   // :213
    if (lprint) printf(" DEP REF  : %g m\n NBINS    : %d\n SIGMIN   : %g\n SIGSTP   : %g\n SIGIN R  : %g\n SIGSTP R : %g\n", zpref, nbins, ds1min, ds1scal, ds1zoom, ds1scalmin);

    std::string cf_vfil = set_file_name(config, tags[0], "V");
    if (chkfile(cf_vfil)) stop(99);
    nc3::Reader v0;
    nc_check(v0.open(cf_vfil), v0.err);
    const int nx = (int)v0.dim_len(cn.x, true), ny = (int)v0.dim_len(cn.y, false), nz = (int)v0.dim_len(cn.z, false);
    if (nx < 1 || ny < 1 || nz < 2) { printf(" ERROR : bad dimensions in %s\n", cf_vfil.c_str()); stop(98); }
    const size_t nxy = (size_t)nx * ny, n3 = nxy * (size_t)nz, n3m = nxy * (size_t)(nz - 1);

    // bin centres, edges and the step -> bin table (:229-262), REAL(8)
    std::vector<double> dsigma(nbins), edge(nbins + 1);
    int ijtrans = 0;
    for (int ji = 1; ji <= nbins; ++ji) {
        const double test = ds1min + ((float)ji - 0.5f) * ds1scal;
        if (test > ds1zoom) { if (!ijtrans) ijtrans = ji; dsigma[ji - 1] = ds1zoom + ((float)(ji - ijtrans) + 0.5f) * ds1scalmin; }
        else dsigma[ji - 1] = test;
    }
    edge[0] = ds1min;
    for (int ji = 2; ji <= nbins; ++ji) edge[ji - 1] = 0.5f * (dsigma[ji - 1] + dsigma[ji - 2]);
    edge[nbins] = edge[nbins - 1] + ds1scalmin;
    const int nsigmax = (int)lround((edge[nbins] - edge[0]) / ds1scalmin);
    if (nsigmax < 1) { printf(" ERROR : empty density axis\n"); stop(99); }
    std::vector<int32_t> itab(nsigmax, 0);
    for (int ji = 1; ji <= nsigmax; ++ji) {
        const double test = ds1min + ((float)ji - 0.5f) * ds1scalmin;
        for (int jj = 1; jj <= nbins; ++jj)
            if (test > edge[jj - 1] && test <= edge[jj]) itab[ji - 1] = jj;
    }
    printf("npiglo = %d\nnpjglo = %d\nnpk    = %d\nnbins  = %d\n", nx, ny, nz, nbins);

    nc3::Reader hgr;
    nc_check(hgr.open(cn.fhgr), hgr.err);
    MeshZgr zgr;
    zgr.open(cn.fzgr);
    std::vector<float> e1v(nxy), e2u(nxy), glamv(nxy), e31d(nz), navlon(nxy, 0.f), navlat(nxy, 0.f);
    read_level(hgr, cn.e1v, 0, 0, nxy, e1v.data());
    read_level(hgr, "e2u", 0, 0, nxy, e2u.data());
    read_level(hgr, "glamv", 0, 0, nxy, glamv.data());
    const bool lperio = nx >= 2 && glamv[0] == glamv[nx - 2];   // :336-337
    if (lfull) read_1d(zgr.nc, zgr.name1d("e3t1d"), nz, e31d.data());
    if (v0.find_var(cn.vlon2d) >= 0) read_level(v0, cn.vlon2d, 0, 0, nxy, navlon.data());
    if (v0.find_var(cn.vlat2d) >= 0) read_level(v0, cn.vlat2d, 0, 0, nxy, navlat.data());
    std::vector<float> e3u, e3v;
    if (!lvvl) {
        e3u.resize(n3); e3v.resize(n3);
        const std::string nu = zgr.ver == "v3.0" ? "e3u" : "e3u_0", nv = zgr.e3v_name();
        for (int k = 0; k < nz; ++k) {
            float *du = e3u.data() + (size_t)k * nxy, *dv = e3v.data() + (size_t)k * nxy;
            if (lfull) for (size_t c = 0; c < nxy; ++c) { du[c] = e31d[k]; dv[c] = e31d[k]; }
            else { read_level(zgr.nc, nu, k, 0, nxy, du); read_level(zgr.nc, nv, k, 0, nxy, dv); }
        }
    }

    gpu_check(cdfgpu_init(-1, 3), "cdfgpu_init");   // the first device, or latitude bands with $CDFGPU_SHARD=lat (frame order kept)
    gpu_check(cdftransig_gpu_setup(nx, ny, nz, nbins, zpref, lteos10 ? 1 : 0, ds1min, ds1scalmin, nsigmax, itab.data(), e2u.data(),
                                   e1v.data(), lvvl ? nullptr : e3u.data(), lvvl ? nullptr : e3v.data(), lperio ? 1 : 0),
              "cdftransig_gpu_setup");
    // two frame slots: one frame read ahead is all the overlap needs (an ORCA12 frame is four 3.97 GB fields)
    const int ns = 2, nbuf = lvvl ? 6 : 4;
    std::vector<std::unique_ptr<Pinned>> pbuf;
    for (int s = 0; s < ns * nbuf; ++s) pbuf.emplace_back(new Pinned(n3));
    // -vvl -full: e3u / e3v filled on the host from e3t1d, once per slot
    if (lvvl && lfull) {
        sibling_host_f32(CDFGPU_CALL_TRANSIG, 4);
        sibling_host_f32(CDFGPU_CALL_TRANSIG, 5);
        for (int s = 0; s < ns; ++s)
            for (int f = 4; f < 6; ++f)
                for (int k = 0; k < nz; ++k) for (size_t c = 0; c < nxy; ++c) pbuf[s * nbuf + f]->p[(size_t)k * nxy + c] = e31d[k];
    }
    tm.mark("setup");
    double dtotal_time = 0.0;
    long nframes = 0;
    for (size_t jtag = 0; jtag < tags.size(); ++jtag) {
        const std::string &tag = tags[jtag];
        if (lprint) printf("  working on  ctag=%s\n", tag.c_str());
        const std::string cf_t = set_file_name(config, tag, "T"), cf_s = lsal ? set_file_name(config, tag, "S") : cf_t;
        const std::string cf_u = set_file_name(config, tag, "U"), cf_v = set_file_name(config, tag, "V");
        bool miss = chkfile(cf_t);
        miss = chkfile(cf_s) || miss; miss = chkfile(cf_u) || miss; miss = chkfile(cf_v) || miss;
        if (miss) stop(99);
        nc3::Reader ft, fs, fu, fv;
        nc_check(ft.open(cf_t), ft.err); nc_check(fs.open(cf_s), fs.err); nc_check(fu.open(cf_u), fu.err); nc_check(fv.open(cf_v), fv.err);
        const int npt = (int)ft.dim_len(cn.t, false);
        { const int it = ft.find_var(cn.vtimec); for (int r = 0; r < npt && it >= 0; ++r) { double x = 0; ft.read_f64(ft.vars[it], r, 0, 1, &x); dtotal_time += x; } }
        // the files of a tag may store a field differently from those of the tag before: declared per tag (the frames of the
        // previous tag still in flight keep the declaration they were submitted with)
        std::vector<RecordField> fields;
        fields.emplace_back(0, fu, "vozocrtx");
        fields.emplace_back(1, fv, cn.vomecrty);
        fields.emplace_back(2, ft, cn.votemper);
        fields.emplace_back(3, fs, cn.vosaline);
        if (lvvl && !lfull) {
            fields.emplace_back(4, fu, "e3u");
            fields.emplace_back(5, fv, "e3v");
        }
        for (auto &f : fields) f.declare_sibling(CDFGPU_CALL_TRANSIG);
        for (int jt = 0; jt < npt; ++jt) {
            const int slot = (int)(nframes % ns);
            if (nframes >= ns) gpu_check(cdftransig_gpu_wait(slot), "cdftransig_gpu_wait");   // the slot's buffers are free again
            float *b[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
            for (int f = 0; f < nbuf; ++f) b[f] = pbuf[slot * nbuf + f]->p;
            for (auto &f : fields) f.read(jt, n3, b[f.field]);
            ++nframes;
            gpu_check(cdftransig_gpu_submit(slot, b[0], b[1], b[2], b[3], b[4], b[5], jtag == 0 ? 1 : 0), "cdftransig_gpu_submit");
        }
    }
    if (nframes == 0) { printf(" ERROR : no time frame in the listed files\n"); stop(99); }
    std::vector<double> du((size_t)nbins * nxy), dv((size_t)nbins * nxy);
    gpu_check(cdftransig_gpu_fetch(du.data(), dv.data()), "cdftransig_gpu_fetch");   // after every frame submitted
    tm.mark("records");
    (void)n3m;

    // CreateOutput (:441-476): create / createvar / putheadervar with cdep = sigma_N and pdep = REAL(dsigma)
    nc3::Writer w;
    const int dx = w.def_dim("x", nx), dy = w.def_dim("y", ny), dz = w.def_dim(clsigma, nbins), dt = w.def_dim("time_counter", 0);
    const int vlon = w.def_var("nav_lon", nc3::NC_FLOAT, {dy, dx}), vlat = w.def_var("nav_lat", nc3::NC_FLOAT, {dy, dx});
    const int vz = w.def_var(clsigma, nc3::NC_FLOAT, {dz}), vt = w.def_var("time_counter", nc3::NC_DOUBLE, {dt});
    const char *names[2] = {"vouxysig", "vovxysig"}, *longn[2] = {"Zonal_trsp_sig_coord", "Meridional_trsp_sig_coord"};
    int vid[2];
    for (int v = 0; v < 2; ++v) {
        vid[v] = w.def_var(names[v], nc3::NC_FLOAT, {dt, dz, dy, dx});
        w.put_att_text(vid[v], "units", "m3/s");
        w.put_att_float(vid[v], "_FillValue", 0.f);
        w.put_att_float(vid[v], "valid_min", -10.f);
        w.put_att_float(vid[v], "valid_max", 10.f);
        w.put_att_text(vid[v], "long_name", longn[v]);
        w.put_att_text(vid[v], "short_name", names[v]);
        w.put_att_int(vid[v], "iweight", (int32_t)nframes);   // putvar(..., kwght=nframes) (:468,472)
        w.put_att_text(vid[v], "online_operation", "N/A");
        w.put_att_text(vid[v], "axis", "TSYX");
    }
    nc_check(w.create(cf_out), w.err);
    w.put_f32(vlon, 0, 0, nxy, navlon.data());
    w.put_f32(vlat, 0, 0, nxy, navlat.data());
    std::vector<float> sig32(nbins);
    for (int b = 0; b < nbins; ++b) sig32[b] = (float)dsigma[b];
    w.put_f32(vz, 0, 0, nbins, sig32.data());
    const double dtimean = dtotal_time / (double)nframes;   // :464
    w.put_f64(vt, 0, 0, 1, &dtimean);
    std::vector<float> plane(nxy);
    for (int v = 0; v < 2; ++v) {
        const std::vector<double> &d = v == 0 ? du : dv;
        for (int b = 0; b < nbins; ++b) {
            for (size_t c = 0; c < nxy; ++c) plane[c] = (float)(d[(size_t)b * nxy + c] / (double)nframes);   // zt = dusigsig(:,:,jk)/nframes
            nc_check(w.put_f32(vid[v], 0, (uint64_t)b * nxy, nxy, plane.data()), w.err);
        }
    }
    w.close();
    tm.mark("output_closed");
    gpu_check(cdfgpu_finalize(), "cdfgpu_finalize");
    tm.total();
    return 0;
}
