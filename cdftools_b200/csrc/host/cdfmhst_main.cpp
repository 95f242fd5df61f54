// cdfmhst_gpu -- C++ twin of the cdfmhst command line (src/cdfmhst.f90) on top of libcdfgpu's C ABI.
// Same options, auxiliary files, output variables (zomht_* [zomst_*]), ASCII tables and exit codes (99 usage / missing
// file / unknown option, 98 NetCDF, 97 GPU library).  The level loop cdfmhst.f90:303-366 (vertical integral of
// vomevt / vomevs * e1v * e3v and the masked zonal sums) is replaced by the record pipeline cdfmhst_gpu_submit, or in -v/-t
// mode cdfmhst_gpu_submit_vts, which also forms the V-point products of :313-323 on the device, and cdfmhst_gpu_fetch; the
// basin combinations, the scaling and the missing-value replacement (:370-441) stay on the host as in the reference.
#include <memory>

#include "host_common.hpp"

using namespace cdfhost;

int main(int argc, char **argv)
{
    PhaseTimer tm("cdfmhst_gpu");
    Names cn;
    if (argc == 1) {
        printf(" usage : cdfmhst_gpu  -vt VT-file | (-v V-file -t T-file [-s S-file]) [-vtvar VT-var VS-var]\n"
               "         [-MST] [-b BASIN-mask] [-full] [-Zdim] [-o OUT-file] [-vvl]\n"
               "     PURPOSE : meridional heat / salt transport as a function of latitude, on a B200 GPU.\n"
               "     REQUIRED FILES : %s, %s and %s ; %s optional (sub-basins)\n"
               "     OUTPUT : mhst.nc (zomht_glo [zomht_atl _inp _ind _pac _inp0] [zomst_*]), zonal_heat_trp.dat, zonal_salt_trp.dat\n",
               cn.fhgr.c_str(), cn.fzgr.c_str(), cn.fmsk.c_str(), cn.fbasins.c_str());
        return 0;
    }
    std::string cf_vtfil = "none", cf_vfil = "none", cf_tfil = "none", cf_sfil = "none", cf_outnc = "mhst.nc";
    std::string cn_vomevt = "vomevt", cn_vomevs = "vomevs";
    int npvar = 1;
    bool lfull = false, lzdim = false, lvvl = false;
    for (int i = 1; i < argc;) {   // cdfmhst.f90:176-194
        const std::string a = argv[i++];
        auto next = [&]() { return std::string(i < argc ? argv[i++] : ""); };
        if (a == "-vt") cf_vtfil = next();
        else if (a == "-vtvar") { cn_vomevt = next(); cn_vomevs = next(); }
        else if (a == "-v") cf_vfil = next();
        else if (a == "-t") cf_tfil = next();
        else if (a == "-s") cf_sfil = next();
        else if (a == "-MST") npvar = 2;
        else if (a == "-full") lfull = true;
        else if (a == "-Zdim") lzdim = true;
        else if (a == "-b") cn.fbasins = next();
        else if (a == "-o") cf_outnc = next();
        else if (a == "-vvl") lvvl = true;
        else { printf(" ERROR : %s : unknown option.\n", a.c_str()); stop(99); }
    }
    const bool lsepf = cf_vtfil == "none";
    bool lchk = false;   // cdfmhst.f90:198-216
    if (lsepf) {
        lchk = chkfile(cf_vfil == "none" ? "(no -vt / -v file)" : cf_vfil) || lchk;
        lchk = chkfile(cf_tfil == "none" ? "(no -t file)" : cf_tfil) || lchk;
        if (lchk) stop(99);
        if (cf_sfil == "none") cf_sfil = cf_tfil;
    }
    lchk = chkfile(cn.fhgr) || lchk; lchk = chkfile(cn.fzgr) || lchk; lchk = chkfile(cn.fmsk) || lchk;
    lchk = chkfile(cf_vtfil) || lchk;
    if (lsepf) { lchk = chkfile(cf_tfil) || lchk; lchk = chkfile(cf_sfil) || lchk; }
    if (lchk) stop(99);
    const bool llglo = !chkfile(cn.fbasins, false);
    if (!llglo) printf(" Only compute for GLOBAL basin\n");
    const int nbasinso = llglo ? 6 : 1;
    if (lsepf) cf_vtfil = cf_vfil;

    nc3::Reader vt;
    nc_check(vt.open(cf_vtfil), vt.err);
    const int nx = (int)vt.dim_len(cn.x, true), ny = (int)vt.dim_len(cn.y, false), nz = (int)vt.dim_len(cn.z, false);
    const int npt = (int)vt.dim_len(cn.t, false);
    printf("npiglo = %d\nnpjglo = %d\nnpk    = %d\nnpt    = %d\n", nx, ny, nz, npt);
    if (nx < 1 || ny < 1 || nz < 1) { printf(" ERROR : bad dimensions in %s\n", cf_vtfil.c_str()); stop(98); }
    const int npko = lzdim ? nz : 1;
    const size_t nxy = (size_t)nx * ny, n3 = nxy * (size_t)nz;

    nc3::Reader hgr, msk;
    nc_check(hgr.open(cn.fhgr), hgr.err);
    nc_check(msk.open(cn.fmsk), msk.err);
    MeshZgr zgr;
    zgr.open(cn.fzgr);
    std::vector<float> e1v(nxy), gphiv(nxy), gdep(npko, 0.f), e31d(nz), navlat, vmask1(nxy), atl, pac, ind;
    read_level(hgr, cn.e1v, 0, 0, nxy, e1v.data());
    read_level(hgr, cn.gphiv, 0, 0, nxy, gphiv.data());
    if (lzdim) read_1d(zgr.nc, zgr.name1d("gdept"), nz, gdep.data());
    if (lfull) read_1d(zgr.nc, zgr.name1d("e3t1d"), nz, e31d.data());
    dummy_lat(gphiv, nx, ny, navlat);
    read_level(msk, cn.vmask, 0, 0, nxy, vmask1.data());
    if (llglo) {
        nc3::Reader bas;
        nc_check(bas.open(cn.fbasins), bas.err);
        atl.resize(nxy); pac.resize(nxy); ind.resize(nxy);
        read_level(bas, cn.tmaskatl, 0, 0, nxy, atl.data());
        read_level(bas, cn.tmaskpac, 0, 0, nxy, pac.data());
        read_level(bas, cn.tmaskind, 0, 0, nxy, ind.data());
    }
    std::vector<float> e3v(n3);
    auto load_e3v = [&](long rec) {   // cdfmhst.f90:331-334 (with -vvl e3v comes from the VT / V file, :218-221)
        nc3::Reader *src = lvvl ? &vt : &zgr.nc;
        const std::string name = lvvl ? "e3v" : zgr.e3v_name();
        for (int k = 0; k < nz; ++k) {
            float *dst = e3v.data() + (size_t)k * nxy;
            if (lfull) for (size_t c = 0; c < nxy; ++c) dst[c] = e31d[k];
            else read_level(*src, name, k, rec, nxy, dst);
        }
    };
    load_e3v(0);

    // CreateOutput (cdfmhst.f90:502-549)
    const char *cbasin[6] = {"_glo", "_atl", "_inp", "_ind", "_pac", "_inp0"};
    const std::string axis = lzdim ? "TZY" : "TY";
    std::vector<OutVar> ovars;
    for (int b = 0; b < nbasinso; ++b)
        ovars.push_back({std::string("zomht") + cbasin[b], std::string("Meridional Heat Transport ") + cbasin[b], "PW", -10.f, 20.f, 9999.99f, axis});
    if (npvar == 2)
        for (int b = 0; b < nbasinso; ++b)
            ovars.push_back({std::string("zomst") + cbasin[b], std::string("Meridional Salt Transport ") + cbasin[b], "T/sec", -10.e9f, 20.e9f, 9999.99f, axis});
    std::vector<double> tim(npt, 0.0);
    { const int it = vt.find_var(cn.vtimec); if (it >= 0) for (int r = 0; r < npt; ++r) vt.read_f64(vt.vars[it], r, 0, 1, &tim[r]); }
    OutFile out;
    out.create(cf_outnc, "depthv", ny, npko, ovars, "", navlat, gdep, tim, vt);
    FILE *fh = fopen("zonal_heat_trp.dat", "w"), *fs = fopen("zonal_salt_trp.dat", "w");
    if (!fh || !fs) { printf(" ERROR : cannot open the ASCII output files\n"); stop(98); }

    gpu_check(cdfgpu_init(-1, 3), "cdfgpu_init");   // $CDFGPU_DEVICES / $CDFGPU_SHARD=time: the slots spread over the devices
    auto setup = [&]() {
        gpu_check(cdfmhst_gpu_setup(nx, ny, nz, e1v.data(), e3v.data(), vmask1.data(), llglo ? atl.data() : nullptr,
                                    llglo ? pac.data() : nullptr, llglo ? ind.data() : nullptr), "cdfmhst_gpu_setup");
    };
    setup();
    // record pipeline: record jt is read into slot jt mod ns while the earlier ones are in flight; -vvl re-runs setup per
    // record, so only one record is in flight.  Record buffers per slot: vomevt, vomevs (-vt mode) or V, T, S (separate
    // files: the device forms the V-point products, cdfmhst_gpu_submit_vts); each field raw when the device can decode it
    const int ns = lvvl ? 1 : cdfgpu_nslots();
    std::vector<std::unique_ptr<Pinned>> pbuf;
    for (int s = 0; s < ns; ++s)
        for (int f = 0; f < 3; ++f) pbuf.emplace_back(new Pinned(f < 2 || lsepf ? n3 : 1));
    nc3::Reader tf, sf;
    std::vector<RecordField> fields;
    if (lsepf) {
        nc_check(tf.open(cf_tfil), tf.err);
        nc_check(sf.open(cf_sfil), sf.err);
        fields.emplace_back(0, vt, cn.vomecrty);
        fields.emplace_back(1, tf, cn.votemper);
        fields.emplace_back(2, sf, cn.vosaline);
    } else {
        fields.emplace_back(0, vt, cn_vomevt);
        fields.emplace_back(1, vt, cn_vomevs);
    }
    for (auto &f : fields) f.declare_sibling(lsepf ? CDFGPU_CALL_MHST_VTS : CDFGPU_CALL_MHST);
    tm.mark("setup");
    std::vector<double> heat((size_t)npko * 4 * ny), salt((size_t)npko * 4 * ny);
    std::vector<float> plane((size_t)npko * ny);
    auto drain = [&](int jt) {
        gpu_check(cdfmhst_gpu_fetch(jt % ns, heat.data(), salt.data()), "cdfmhst_gpu_fetch");
        // variables: glo, atl, inp = ind + pac, ind, pac, inp0 = glo - atl; / 1.d15 (PW) or 1.d6; 0 -> ppspval (:384-441)
        for (int v = 0; v < npvar; ++v) {
            const std::vector<double> &d = v == 0 ? heat : salt;
            const double scale = v == 0 ? 1.e15 : 1.e6;
            for (int b = 0; b < nbasinso; ++b) {
                for (int l = 0; l < npko; ++l)
                    for (int j = 0; j < ny; ++j) {
                        const double *q = d.data() + (size_t)l * 4 * ny;   // [m][j]: glo, atl, pac, ind
                        const double glo = q[j], at = q[ny + j], pa = q[2 * ny + j], in = q[3 * ny + j];
                        double x = b == 0 ? glo : b == 1 ? at : b == 2 ? (in + pa) : b == 3 ? in : b == 4 ? pa : (glo - at);
                        x = x / scale;
                        if (x == 0.0) x = (double)9999.99f;
                        plane[(size_t)l * ny + j] = (float)x;
                    }
                out.put(v * nbasinso + b, jt, plane.data());
            }
        }
        // ASCII tables (cdfmhst.f90:447-491, formats 9000 / 9001), values after the last level
        const double *hq = heat.data() + (size_t)(npko - 1) * 4 * ny, *sq = salt.data() + (size_t)(npko - 1) * 4 * ny;
        fprintf(fh, " ! Zonal heat transport (integrated alon I-model coordinate) (in Pw)\n");
        fprintf(fs, "  ! Zonal salt transport (integrated alon I-model coordinate) (in 10^6 kg/s)\n");
        if (llglo) {
            fprintf(fh, " ! J        Global          Atlantic         Pacific          Indian           Mediteranean     Austral  \n");
            fprintf(fs, "  ! J        Global          Atlantic         Pacific          Indian           Mediteranean     Austral  \n");
        } else {
            fprintf(fh, " ! J        Global        \n");
            fprintf(fs, "  J        Global  \n");
        }
        fprintf(fh, "  ! time : %12d\n", jt + 1);
        fprintf(fs, "  ! time : %12d\n", jt + 1);
        for (int j = ny - 1; j >= 0; --j) {
            fprintf(fh, "%4d", j + 1);
            fprintf(fs, "%4d", j + 1);
            const int nm = llglo ? 6 : 1;
            for (int m = 0; m < nm; ++m) {   // glo, atl, pac, ind, med (0), aus (0)
                const double hv = m < 4 ? hq[(size_t)m * ny + j] / 1e15 : 0.0, sv = m < 4 ? sq[(size_t)m * ny + j] / 1e6 : 0.0;
                if (m == 0) { fprintf(fh, " %9.3f %8.4f", navlat[j], hv); fprintf(fs, " %9.2f %9.3f", navlat[j], sv); }
                else { fprintf(fh, " %9.3f", hv); fprintf(fs, " %9.2f", sv); }
            }
            fprintf(fh, "\n");
            fprintf(fs, "\n");
        }
    };
    for (int jt = 0; jt < npt; ++jt) {
        const int slot = jt % ns;
        if (jt >= ns) drain(jt - ns);
        if (lvvl && jt > 0) { load_e3v(jt); setup(); }
        float *b[3] = {pbuf[slot * 3]->p, pbuf[slot * 3 + 1]->p, pbuf[slot * 3 + 2]->p};
        for (auto &f : fields) f.read(jt, n3, b[f.field]);
        if (lsepf)   // temperature / salinity at V points times V, REAL(4), row npjglo = 0 (cdfmhst.f90:313-323), on the device
            gpu_check(cdfmhst_gpu_submit_vts(slot, b[0], b[1], b[2], lzdim ? 1 : 0), "cdfmhst_gpu_submit_vts");
        else
            gpu_check(cdfmhst_gpu_submit(slot, b[0], b[1], lzdim ? 1 : 0), "cdfmhst_gpu_submit");
    }
    for (int jt = npt > ns ? npt - ns : 0; jt < npt; ++jt) drain(jt);
    tm.mark("records");
    fclose(fh);
    fclose(fs);
    out.w.close();
    tm.mark("output_closed");
    gpu_check(cdfgpu_finalize(), "cdfgpu_finalize");
    tm.total();
    return 0;
}
