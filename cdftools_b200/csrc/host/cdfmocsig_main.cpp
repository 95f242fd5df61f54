// cdfmocsig_gpu -- C++ twin of the cdfmocsig command line (src/cdfmocsig.f90) on top of libcdfgpu's C ABI.
// Same options and rules (exactly three mandatory arguments -v -t and -r|-ntr; the default bins are used unless
// ALL of -sigmin -sigstp -nbins are given, cdfmocsig.f90:237,265), same auxiliary files, same output variables.
// The loop nest cdfmocsig.f90:366-475 (missing-value scrub, area, EOS, bin, scatter-add, bin cumsum) is one fused
// kernel per record behind cdfmocsig_gpu_submit / cdfmocsig_gpu_fetch; -isodep (:423-469) adds the zoiso* variables.
#include <array>

#include "host_common.hpp"

using namespace cdfhost;

int main(int argc, char **argv)
{
    Names cn;
    if (argc == 1) {
        printf(" usage : cdfmocsig_gpu  -v V-file -t T-file -r REF-depth | -ntr [-eiv] [-full] ...\n"
               "        ... [-sigmin sigmin] [-sigstp sigstp] [-nbins nbins] [-isodep] ...\n"
               "        ... [-s S-file ] [-o OUT-file] [-vvl] [-verbose] [-teos10] [-nc4]\n");
        return 0;
    }
    PhaseTimer tm("cdfmocsig_gpu");
    CudaWarmup warm;   // CUDA contexts come up while the mesh and mask files are read
    std::string cf_vfil, cf_tfil, cf_sfil = "none", cf_moc = "mocsig.nc", cglobal = "Partial step computation";
    float pref = 0.f, sigmin = 0.f, sigstp = 0.f;
    int nbins = 0, ii = 0;
    bool lbin[3] = {true, true, true}, lntr = false, lfull = false, leiv = false, lvvl = false, lteos10 = false,
         lisodep = false, lprint = false;
    for (int i = 1; i < argc;) {   // cdfmocsig.f90:187-208
        const std::string a = argv[i++];
        auto next = [&]() { return std::string(i < argc ? argv[i++] : ""); };
        if (a == "-v") { cf_vfil = next(); ++ii; }
        else if (a == "-t") { cf_tfil = next(); ++ii; }
        else if (a == "-r") { pref = (float)atof(next().c_str()); ++ii; }
        else if (a == "-ntr") { lntr = true; ++ii; }
        else if (a == "-s") cf_sfil = next();
        else if (a == "-full") { lfull = true; cglobal = "Full step computation"; }
        else if (a == "-eiv") leiv = true;
        else if (a == "-sigmin") { sigmin = (float)atof(next().c_str()); lbin[0] = false; }
        else if (a == "-nbins") { nbins = atoi(next().c_str()); lbin[1] = false; }
        else if (a == "-sigstp") { sigstp = (float)atof(next().c_str()); lbin[2] = false; }
        else if (a == "-o") cf_moc = next();
        else if (a == "-vvl") lvvl = true;
        else if (a == "-teos10") lteos10 = true;
        else if (a == "-isodep") lisodep = true;
        else if (a == "-verbose") lprint = true;
        else if (a == "-nc4") note_nc4();   // DEV_TOOLS/tagnc4.tpl:1-13
        else { printf("  ERROR : %s : unknown option.\n", a.c_str()); stop(99); }
    }
    if (ii != 3) { printf("  ERROR : mandatory arguments missing, see usage please !\n"); stop(99); }
    if (cf_sfil == "none") cf_sfil = cf_tfil;
    bool lchk = false;   // cdfmocsig.f90:218-224
    for (const std::string *f : {&cn.fhgr, &cn.fzgr, &cn.fmsk, &cf_vfil, &cf_tfil, &cf_sfil}) lchk = chkfile(*f) || lchk;
    if (lchk) stop(99);

    nc3::Reader vf, tf, sf;
    nc_check(vf.open(cf_vfil), vf.err);
    nc_check(tf.open(cf_tfil), tf.err);
    nc_check(sf.open(cf_sfil), sf.err);
    const float zsps = sf.spval(var_or_die(sf, cn.vosaline), cn.missing);   // cdfmocsig.f90:227-229
    const float zspt = tf.spval(var_or_die(tf, cn.votemper), cn.missing);
    const float zspv = vf.spval(var_or_die(vf, cn.vomecrty), cn.missing);
    const bool ldefault_bins = lbin[0] || lbin[1] || lbin[2];   // :237
    const int nx = (int)vf.dim_len(cn.x, true), ny = (int)vf.dim_len(cn.y, false), nz = (int)vf.dim_len(cn.z, false);
    const int npt = (int)vf.dim_len(cn.t, false);
    printf("npiglo = %d\nnpjglo = %d\nnpk    = %d\nnpt    = %d\n", nx, ny, nz, npt);
    const bool lbas = !chkfile(cn.fbasins, false);
    const int nb = lbas ? 5 : 1;
    if (ldefault_bins) {   // :265-292
        if (lntr) { nbins = 52; sigmin = 1023.f; sigstp = 0.1f; }
        else switch ((int)pref) {
            case 0: nbins = 52; sigmin = 23.f; sigstp = 0.1f; break;
            case 1000: nbins = 88; sigmin = 24.f; sigstp = 0.1f; break;
            case 2000: nbins = 158; sigmin = 30.f; sigstp = 0.05f; break;
            default:
                printf(" This value of depth_ref (%g) is not implemented as standard\n You must use the -sigmin, -sigstp and -nbins options to precise\n the density bining you want to use.\n", pref);
                stop(99);
        }
    }
    if (lntr) printf("  For Neutral density MOC\n"); else printf("  For reference depth %6.1f m, \n", pref);
    printf("  You are using -sigmin %5.2f -sigstp %5.2f -nbins %3d\n", sigmin, sigstp, nbins);
    std::vector<float> sigma(nbins);   // :302-304, REAL(4) arithmetic
    for (int n = 1; n <= nbins; ++n) { volatile float t = (float)n - 0.5f; t = t * sigstp; sigma[n - 1] = sigmin + t; }
    if (lprint) printf("  min density: %g  max density: %g\n", sigma[0], sigma[nbins - 1]);

    const size_t nxy = (size_t)nx * ny, n3 = nxy * (size_t)(nz - 1);
    nc3::Reader hgr;
    nc_check(hgr.open(cn.fhgr), hgr.err);
    MeshZgr zgr;
    zgr.open(cn.fzgr);
    std::vector<float> e1v(nxy), gphiv(nxy), e31d(nz), navlat(ny, 0.f);
    read_level(hgr, cn.e1v, 0, 0, nxy, e1v.data());
    if (lfull) read_1d(zgr.nc, zgr.name1d("e3t1d"), nz, e31d.data());
    if (ny > 1) { read_level(hgr, cn.gphiv, 0, 0, nxy, gphiv.data()); dummy_lat(gphiv, nx, ny, navlat); }   // :331-337
    std::vector<int16_t> ibmask;
    basin_masks(cn, lbas, nx, ny, lbas, ibmask);   // the edge zeroing sits inside IF(lbas) here (:349-359)

    // e3v per level, NOT masked (:387-390); with -vvl it comes from the V file per record
    std::vector<float> e3v;
    if (!lvvl) {
        e3v.resize(nxy * (nz - 1));
        for (int k = 0; k < nz - 1; ++k) {
            float *dst = e3v.data() + (size_t)k * nxy;
            if (lfull) for (size_t c = 0; c < nxy; ++c) dst[c] = e31d[k];
            else read_level(zgr.nc, zgr.e3v_name(), k, 0, nxy, dst);
        }
    }

    const char *bn[5] = {"glo", "atl", "inp", "ind", "pac"};
    const char *ln[5] = {"Global", "Atlantic", "IndoPacif", "Indian", "pacif"};
    std::vector<OutVar> ovars;
    for (int b = 0; b < nb; ++b)
        ovars.push_back({std::string("zomsf") + bn[b], std::string("Meridional_Overt.Cell_") + ln[b], "Sverdrup", -1000.f, 1000.f});
    if (lisodep)   // cdfmocsig.f90:537-574
        for (int b = 0; b < nb; ++b)
            ovars.push_back({std::string("zoiso") + bn[b], std::string("Zonal_mean_isopycnal_depth_") + ln[b], "m", 0.f, 8000.f});
    std::vector<double> tim(npt, 0.0);
    { const int it = vf.find_var(cn.vtimec); if (it >= 0) for (int r = 0; r < npt; ++r) vf.read_f64(vf.vars[it], r, 0, 1, &tim[r]); }
    OutFile out;
    out.create(cf_moc, "sigma", ny, nbins, ovars, cglobal + " cdfmocsig", navlat, sigma, tim, vf);

    const int eos = lntr ? CDFGPU_EOS_NEUTRAL : (lteos10 ? CDFGPU_EOS_TEOS10 : CDFGPU_EOS_EOS80);
    tm.mark("mesh_mask_read");
    warm.join();
    gpu_check(cdfgpu_init(-1, 3), "cdfgpu_init");   // $CDFGPU_DEVICES / $CDFGPU_SHARD: several devices behind the same calls
    tm.mark("cuda_init_wait");
    gpu_check(cdfmocsig_gpu_setup(nx, ny, nz, nb, nbins, sigmin, sigstp, pref, eos, e1v.data(), lvvl ? nullptr : e3v.data(),
                                  ibmask.data(), zspv, zspt, zsps, 0, ny), "cdfmocsig_gpu_setup");
    if (lisodep) {   // gdep(:) = -getvare3(cn_fzgr, cn_gdept, npk) is formed inside the library (cdfmocsig.f90:328)
        std::vector<float> gdept(nz);
        read_1d(zgr.nc, zgr.name1d("gdept"), nz, gdept.data());
        gpu_check(cdfmocsig_gpu_set_isodep(gdept.data()), "cdfmocsig_gpu_set_isodep");
    }
    std::vector<RecordField> fields;   // the record arrays of cdfmocsig_gpu_submit: 0 zv, 1 zt, 2 zs, 3 zveiv, 4 e3v_vvl
    fields.emplace_back(0, vf, cn.vomecrty);
    fields.emplace_back(1, tf, cn.votemper);
    fields.emplace_back(2, sf, cn.vosaline);
    if (leiv) fields.emplace_back(3, vf, cn.vomeeivv);
    if (lvvl) fields.emplace_back(4, vf, "e3v");
    declare_submit(fields);

    tm.mark("gpu_setup");
    // -vvl rebuilds the resident area field per record: one record per device in flight
    const int nslot = lvvl ? std::max(1, cdfgpu_nslots() / 3) : cdfgpu_nslots();
    std::vector<std::array<Pinned *, 5>> pbuf(nslot);   // [slot][field], null for an array the run does not pass
    for (auto &b : pbuf)
        for (auto &f : fields) b[f.field] = new Pinned(n3);
    auto buf = [&](int slot, int field) -> float * { return pbuf[slot][field] ? pbuf[slot][field]->p : nullptr; };
    std::vector<double> dmoc((size_t)nb * nbins * ny);
    std::vector<float> plane((size_t)nbins * ny);
    auto drain = [&](int slot, int jt) {   // :478-483
        gpu_check(cdfmocsig_gpu_fetch(slot, dmoc.data()), "cdfmocsig_gpu_fetch");
        for (int b = 0; b < nb; ++b) {
            for (int n = 0; n < nbins; ++n) for (int j = 0; j < ny; ++j) plane[(size_t)n * ny + j] = (float)dmoc[((size_t)j * nbins + n) * nb + b];
            out.put(b, jt, plane.data());
        }
        if (lisodep) {
            gpu_check(cdfmocsig_gpu_fetch_isodep(slot, dmoc.data()), "cdfmocsig_gpu_fetch_isodep");
            for (int b = 0; b < nb; ++b) {
                for (int n = 0; n < nbins; ++n) for (int j = 0; j < ny; ++j) plane[(size_t)n * ny + j] = (float)dmoc[((size_t)j * nbins + n) * nb + b];
                out.put(nb + b, jt, plane.data());
            }
        }
    };
    for (int jt = 0; jt < npt; ++jt) {   // :361
        const int slot = jt % nslot;
        if (jt >= nslot) drain(slot, jt - nslot);
        if (lprint) printf(" working at record %d\n", jt + 1);
        for (auto &f : fields) f.read(jt, n3, buf(slot, f.field));
        gpu_check(cdfmocsig_gpu_submit(slot, jt, buf(slot, 0), buf(slot, 1), buf(slot, 2), buf(slot, 3), buf(slot, 4)),
                  "cdfmocsig_gpu_submit");
    }
    for (int jt = (npt > nslot ? npt - nslot : 0); jt < npt; ++jt) drain(jt % nslot, jt);
    tm.mark("records");
    out.w.close();
    tm.mark("output_closed");
    if (quick_exit_wanted()) { tm.total(); quick_exit_now(); }
    for (auto &b : pbuf) for (auto p : b) delete p;
    gpu_check(cdfgpu_finalize(), "cdfgpu_finalize");
    tm.mark("teardown");
    tm.total();
    return 0;
}
