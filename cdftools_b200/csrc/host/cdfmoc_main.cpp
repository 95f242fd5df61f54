// cdfmoc_gpu -- C++ twin of the cdfmoc command line (src/cdfmoc.f90) on top of libcdfgpu's C ABI.
// Same options, same auxiliary files in the CWD (or CDFT_* environment), same output variables and attributes,
// same exit codes (STOP 99: usage / missing file / unknown option; 98: NetCDF; new 97: GPU library error).
// The hot loop nest cdfmoc.f90:352-388 is replaced by cdfmoc_gpu_submit / cdfmoc_gpu_fetch with a 3-deep record
// pipeline: record jt+1 is read and sent to the device while record jt is being integrated.
// -decomp (cdfmoc.f90:390-517) runs on the GPU too (one record in flight); -rapid (:598-1004) stays with the
// Fortran host (an O(nx*nz) section diagnostic, not part of the hot path).
#include "host_common.hpp"

using namespace cdfhost;

static void usage(const Names &cn)
{
    printf(" usage : cdfmoc_gpu  -v V-file [-t T-file] [-s S-file] [-u U-file] [-o OUT-file] [-full] [-decomp] [-rapid] [-vvl] [-teos10] [-nc4]\n"
           "      \n     PURPOSE :\n"
           "       Compute the Meridional Overturning Cell (MOC) on a B200 GPU: zonal integral of the\n"
           "       meridional transport for every basin, integrated from the bottom (Sv).\n"
           "     REQUIRED FILES :\n        %s, %s, %s ; %s is optional (sub-basins)\n"
           "     OUTPUT : netcdf file moc.nc, variables zomsfglo [zomsfatl zomsfinp zomsfind zomsfpac zomsfinp0]\n",
           cn.fhgr.c_str(), cn.fzgr.c_str(), cn.fmsk.c_str(), cn.fbasins.c_str());
}

int main(int argc, char **argv)
{
    Names cn;
    if (argc == 1) { usage(cn); return 0; }   // the reference prints the usage and STOPs (cdfmoc.f90:129-209)
    PhaseTimer tm("cdfmoc_gpu");
    CudaWarmup warm;   // CUDA contexts come up while the mesh and mask files are read
    std::string cf_vfil, cf_tfil = "none", cf_sfil = "none", cf_ufil = "none", cf_moc = "moc.nc";
    std::string cglobal = "Partial step computation";
    bool lfull = false, ldec = false, lrap = false, lvvl = false, lteos10 = false;
    for (int i = 1; i < argc;) {   // cdfmoc.f90:217-234
        const std::string a = argv[i++];
        auto next = [&]() { return std::string(i < argc ? argv[i++] : ""); };
        if (a == "-v") cf_vfil = next();
        else if (a == "-t") cf_tfil = next();
        else if (a == "-s") cf_sfil = next();
        else if (a == "-u") cf_ufil = next();
        else if (a == "-o") cf_moc = next();
        else if (a == "-full") { lfull = true; cglobal = "Full step computation"; }
        else if (a == "-decomp") ldec = true;
        else if (a == "-rapid") lrap = true;
        else if (a == "-vvl") lvvl = true;
        else if (a == "-teos10") lteos10 = true;
        else if (a == "-nc4") note_nc4();   // DEV_TOOLS/tagnc4.tpl:1-13
        else { printf("  ERROR : %s : unknown option.\n", a.c_str()); stop(99); }
    }
    (void)lteos10; (void)cf_ufil;
    if (cf_sfil == "none") cf_sfil = cf_tfil;
    bool lchk = false;   // cdfmoc.f90:240-246
    lchk = chkfile(cn.fhgr) || lchk; lchk = chkfile(cn.fzgr) || lchk; lchk = chkfile(cn.fmsk) || lchk;
    lchk = chkfile(cf_vfil.empty() ? "(no -v file)" : cf_vfil) || lchk;
    if (ldec || lrap) lchk = chkfile(cf_tfil) || chkfile(cf_sfil) || lchk;
    if (lchk) stop(99);
    if (lrap) {
        printf(" ERROR : -rapid is not part of the GPU hot path; use the Fortran host for it.\n");
        stop(99);
    }

    nc3::Reader vf;
    nc_check(vf.open(cf_vfil), vf.err);
    const int nx = (int)vf.dim_len(cn.x, true), ny = (int)vf.dim_len(cn.y, false), nz = (int)vf.dim_len(cn.z, false);
    const int npt = (int)vf.dim_len(cn.t, false);
    printf(" Working with cdfmoc ...\n   npiglo = %d\n   npjglo = %d\n   npk    = %d\n   npt    = %d\n", nx, ny, nz, npt);
    if (nx < 1 || ny < 1 || nz < 2) { printf(" ERROR : bad dimensions in %s\n", cf_vfil.c_str()); stop(98); }
    const bool lbas = !chkfile(cn.fbasins, false);   // cdfmoc.f90:270-274
    const int nb = lbas ? 5 : 1;
    const size_t nxy = (size_t)nx * ny, n3 = nxy * (size_t)(nz - 1);

    nc3::Reader hgr;
    nc_check(hgr.open(cn.fhgr), hgr.err);
    MeshZgr zgr;
    zgr.open(cn.fzgr);
    std::vector<float> e1v(nxy), gphiv(nxy), gdepw(nz), e31d(nz), navlat;
    read_level(hgr, cn.e1v, 0, 0, nxy, e1v.data());
    read_level(hgr, cn.gphiv, 0, 0, nxy, gphiv.data());
    read_1d(zgr.nc, zgr.name1d("gdepw"), nz, gdepw.data());
    for (auto &d : gdepw) d = -1.f * d;   // cdfmoc.f90:309
    if (lfull) read_1d(zgr.nc, zgr.name1d("e3t1d"), nz, e31d.data());
    dummy_lat(gphiv, nx, ny, navlat);

    std::vector<int16_t> ibmask;
    basin_masks(cn, lbas, nx, ny, true, ibmask);

    // e3v(:,:,jk) = get_e3v(jk,it) = e3v_file * ivmask (cdfmoc.f90:343-348,590-594)
    nc3::Reader msk;
    nc_check(msk.open(cn.fmsk), msk.err);
    std::vector<float> e3v(nxy * nz), lev(nxy);
    auto load_e3v = [&](long rec) {
        nc3::Reader *src = lvvl ? &vf : &zgr.nc;
        const std::string name = lvvl ? cn.ve3vvvl : zgr.e3v_name();
        for (int k = 0; k < nz; ++k) {
            float *dst = e3v.data() + (size_t)k * nxy;
            if (lfull) for (size_t c = 0; c < nxy; ++c) dst[c] = e31d[k];
            else read_level(*src, name, k, rec, nxy, dst);
            read_level(msk, cn.vmask, k, 0, nxy, lev.data());
            for (size_t c = 0; c < nxy; ++c) dst[c] = dst[c] * (float)(int16_t)lev[c];
        }
    };
    load_e3v(0);

    // output file (CreateOutput, cdfmoc.f90:1006-1188)
    // variable order of CreateOutput (cdfmoc.f90:1030-1180): per basin total [, _sh, _bt, _ag], then inp0 likewise
    const char *vn[6] = {"zomsfglo", "zomsfatl", "zomsfinp", "zomsfind", "zomsfpac", "zomsfinp0"};
    const char *vl[6] = {"Global", "Atlantic", "IndoPacif", "Indian", "pacif", "IndPac0"};
    const char *dsuf[3] = {"_sh", "_bt", "_ag"};
    // long names as the reference spells them (cdfmoc.f90:1041-1176): "Ageostoph" for the global cell only, "_Pacif" in the
    // components of the Pacific cell
    const char *dlong[3] = {"GeoShear_Merid_StreamFunction", "Barotropic_Merid_StreamFunction", "Ageostroph_Merid_StreamFunction"};
    const char *vld[6] = {"Global", "Atlantic", "IndoPacif", "Indian", "Pacif", "IndPac0"};
    std::vector<OutVar> ovars;
    for (int b = 0; b < (lbas ? 6 : 1); ++b) {
        ovars.push_back({vn[b], std::string("Meridional_Overt.Cell_") + vl[b], "Sverdrup", -1000.f, 1000.f});
        if (ldec)
            for (int d = 0; d < 3; ++d)
                ovars.push_back({std::string(vn[b]) + dsuf[d],
                                 b ? std::string(dlong[d]) + "_" + vld[b] : std::string(d == 2 ? "Ageostoph_Merid_StreamFunction" : dlong[d]),
                                 "Sverdrup", -1000.f, 1000.f});
    }
    std::vector<double> tim(npt, 0.0);
    { const int it = vf.find_var(cn.vtimec); if (it >= 0) for (int r = 0; r < npt; ++r) vf.read_f64(vf.vars[it], r, 0, 1, &tim[r]); }
    OutFile out;
    out.create(cf_moc, cn.vdepthw, ny, nz, ovars, cglobal, navlat, gdepw, tim, vf);

    tm.mark("mesh_mask_read");
    // ---- GPU: setup once, then the record pipeline
    warm.join();
    gpu_check(cdfgpu_init(-1, 3), "cdfgpu_init");   // $CDFGPU_DEVICES / $CDFGPU_SHARD: several devices behind the same calls
    tm.mark("cuda_init_wait");
    gpu_check(cdfmoc_gpu_setup(nx, ny, nz, nb, e1v.data(), e3v.data(), ibmask.data()), "cdfmoc_gpu_setup");
    std::vector<RecordField> fields;   // the record arrays of the submit call: 0 zv [, 1 zt, 2 zs with -decomp]
    fields.emplace_back(0, vf, cn.vomecrty);
    if (ldec) {   // extra fields of the decomposition (cdfmoc.f90:312-313,439-442)
        std::vector<float> e1u(nxy), gdept(nz);
        read_level(hgr, cn.e1u, 0, 0, nxy, e1u.data());
        read_1d(zgr.nc, zgr.name1d("gdept"), nz, gdept.data());
        std::vector<int16_t> um(n3), tm(n3);
        for (int k = 0; k < nz - 1; ++k) {
            read_level(msk, cn.umask, k, 0, nxy, lev.data());
            for (size_t c = 0; c < nxy; ++c) um[(size_t)k * nxy + c] = (int16_t)lev[c];
            read_level(msk, cn.tmask, k, 0, nxy, lev.data());
            for (size_t c = 0; c < nxy; ++c) tm[(size_t)k * nxy + c] = (int16_t)lev[c];
        }
        gpu_check(cdfmoc_gpu_decomp_setup(lteos10 ? 1 : 0, e1u.data(), gphiv.data(), gdept.data(), um.data(), tm.data()),
                  "cdfmoc_gpu_decomp_setup");
    }
    tm.mark("gpu_setup");
    // record slots: 3 per device under time sharding (every device has its own pipeline), 3 otherwise; -vvl rebuilds the
    // resident area field per record, so only one record per device is in flight
    const int ndev = cdfgpu_num_devices();
    const int ns = (lvvl || ldec) ? ((lvvl && !ldec) ? std::max(1, cdfgpu_nslots() / 3) : 1) : cdfgpu_nslots();
    (void)ndev;
    std::vector<Pinned *> pbuf;
    for (int s = 0; s < std::max(ns, 3); ++s) pbuf.push_back(new Pinned(n3));
    std::vector<float *> bufs;
    for (auto p : pbuf) bufs.push_back(p->p);
    std::vector<double> dmoc((size_t)nb * ny * nz);
    std::vector<float> plane((size_t)nz * ny);
    auto drain = [&](int slot, int jt) {   // cdfmoc.f90:520-551
        gpu_check(cdfmoc_gpu_fetch(slot, dmoc.data()), "cdfmoc_gpu_fetch");
        for (int b = 0; b < nb; ++b) {
            for (int k = 0; k < nz; ++k) for (int j = 0; j < ny; ++j) plane[(size_t)k * ny + j] = (float)dmoc[((size_t)k * ny + j) * nb + b];
            out.put(b, jt, plane.data());
        }
        if (lbas) {
            for (int k = 0; k < nz; ++k) for (int j = 0; j < ny; ++j) {
                const size_t o = ((size_t)k * ny + j) * nb;
                plane[(size_t)k * ny + j] = (float)(dmoc[o + 0] - dmoc[o + 1]);
            }
            out.put(nb, jt, plane.data());
        }
    };
    nc3::Reader tf, sf;
    if (ldec) {   // T and S of the record (cdfmoc.f90:441-442)
        nc_check(tf.open(cf_tfil), tf.err);
        nc_check(sf.open(cf_sfil), sf.err);
        fields.emplace_back(1, tf, cn.votemper);
        fields.emplace_back(2, sf, cn.vosaline);
    }
    declare_submit(fields);
    if (ldec) {   // one record in flight; V, T, S of the record (cdfmoc.f90:357,441-442)
        std::vector<double> dsh(dmoc.size()), dbt(dmoc.size()), dag(dmoc.size());
        const std::vector<double> *comp[4] = {&dmoc, &dsh, &dbt, &dag};
        for (int jt = 0; jt < npt; ++jt) {
            if (lvvl && jt > 0) { load_e3v(jt); gpu_check(cdfmoc_gpu_set_e3v(e3v.data()), "cdfmoc_gpu_set_e3v"); }
            for (auto &f : fields) f.read(jt, n3, bufs[f.field]);
            gpu_check(cdfmoc_gpu_decomp_submit(0, jt, bufs[0], bufs[1], bufs[2]), "cdfmoc_gpu_decomp_submit");
            gpu_check(cdfmoc_gpu_decomp_fetch(0, dmoc.data(), dsh.data(), dbt.data(), dag.data()), "cdfmoc_gpu_decomp_fetch");
            int iv = 0;
            for (int b = 0; b < (lbas ? 6 : 1); ++b)
                for (int d = 0; d < 4; ++d, ++iv) {
                    const std::vector<double> &a = *comp[d];
                    for (int k = 0; k < nz; ++k) for (int j = 0; j < ny; ++j) {
                        const size_t o = ((size_t)k * ny + j) * nb;
                        plane[(size_t)k * ny + j] = (b < 5) ? (float)a[o + b] : (float)(a[o + 0] - a[o + 1]);   // inp0 = glo - atl (:549-566)
                    }
                    out.put(iv, jt, plane.data());
                }
        }
        out.w.close();
        gpu_check(cdfgpu_finalize(), "cdfgpu_finalize");
        return 0;
    }
    for (int jt = 0; jt < npt; ++jt) {   // cdfmoc.f90:338
        const int slot = lvvl ? 0 : jt % ns;
        if (!lvvl && jt >= ns) drain(slot, jt - ns);
        if (lvvl && jt > 0) { load_e3v(jt); gpu_check(cdfmoc_gpu_set_e3v(e3v.data()), "cdfmoc_gpu_set_e3v"); }
        fields[0].read(jt, n3, bufs[slot]);   // zv, the one field without -decomp
        gpu_check(cdfmoc_gpu_submit(slot, jt, bufs[slot]), "cdfmoc_gpu_submit");
        if (lvvl) drain(slot, jt);   // -vvl: the area field changes per record, so only one record is in flight
    }
    if (!lvvl) for (int jt = (npt > ns ? npt - ns : 0); jt < npt; ++jt) drain(jt % ns, jt);
    tm.mark("records");
    out.w.close();
    tm.mark("output_closed");
    if (quick_exit_wanted()) { tm.total(); quick_exit_now(); }
    for (auto p : pbuf) delete p;
    gpu_check(cdfgpu_finalize(), "cdfgpu_finalize");
    tm.mark("teardown");
    tm.total();
    return 0;
}
