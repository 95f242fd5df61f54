// cdfsigtrp_gpu -- C++ twin of the cdfsigtrp command line (src/cdfsigtrp.f90) on top of libcdfgpu.
// Same required arguments (-t -u -v -smin -smax -nbins) and options -s, -full, -refdep, -neutral, -section, -temp, -teos10,
// -help; the same section file (pairs of lines: name [suffix] [long-name prefix] / imin imax jmin jmax, closed by EOF), the
// same outputs (trpsig.txt, <section>_trpsig.nc | _trptemp.nc) and exit codes (99 usage / missing file, 98 NetCDF, 97 GPU
// library).  The section slices are read and prepared here as at :404-555; the loop nests :559-627 run on the device
// (cdfsigtrp_gpu_section).  -brk (a broken-line file of cdf_xtrac_brokenline as one pseudo-zonal section, :465-495), -print
// (the tables of print_out, :902-963) and -xtra (<section>_secdep.nc, <section>_secsig.nc: cdf_writ, :750-900) are host-side
// and implemented here.  Not in this twin: -vvl, and -full together with -brk -- refused with a message.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <memory>

#include "host_common.hpp"

using namespace cdfhost;

struct Section {
    std::string name, varname = "none", longname = "none";
    int imin = 0, imax = 0, jmin = 0, jmax = 0;
};

// section_init (:680-748): name lines are cut at single blanks into at most three words; a line holding EOF ends the list
static std::vector<Section> section_init(const std::string &path)
{
    std::ifstream f(path);
    std::vector<Section> out;
    std::string line;
    while (std::getline(f, line)) {
        if (line.find("EOF") != std::string::npos) break;
        Section s;
        std::string w[3] = {"none", "none", "none"};
        int n = 0;
        std::string rest = line + " ";
        size_t ipos = rest.find(' ');
        while (ipos != std::string::npos && ipos >= 1 && n < 3) {   // INDEX(cline,' ') > 1
            w[n++] = rest.substr(0, ipos);
            rest = rest.substr(ipos + 1);
            ipos = rest.find(' ');
        }
        s.name = w[0]; s.varname = w[1]; s.longname = w[2];
        if (!std::getline(f, line)) { printf(" ERROR : %s : section %s has no position line\n", path.c_str(), s.name.c_str()); stop(99); }
        if (sscanf(line.c_str(), "%d %d %d %d", &s.imin, &s.imax, &s.jmin, &s.jmax) != 4) {
            printf(" ERROR : %s : cannot read imin imax jmin jmax of section %s\n", path.c_str(), s.name.c_str());
            stop(99);
        }
        out.push_back(s);
    }
    return out;
}

struct Field {   // one (t,z,y,x) variable of an open file
    nc3::Reader *nc = nullptr;
    const nc3::Var *v = nullptr;
    int nx = 0, ny = 0;
    Field(nc3::Reader &r, const std::string &var, const Names &cn) : nc(&r), v(&var_or_die(r, var))
    {
        nx = (int)r.dim_len(cn.x, true);
        ny = (int)r.dim_len(cn.y, false);
    }
    // getvarxz (cdfio.F90:1950-2043): out[k][0..npts) = var(kimin : kimin+npts-1, kj, k), first time frame
    void xz(int kj, int npts, int npk, int kimin, float *out) const
    {
        for (int k = 0; k < npk; ++k)
            nc_check(nc->read_f32(*v, 0, ((uint64_t)k * ny + (kj - 1)) * nx + (kimin - 1), npts, out + (size_t)k * npts), nc->err);
    }
    // getvaryz (cdfio.F90:2046-2148): out[k][0..npts) = var(ki, kjmin : kjmin+npts-1, k)
    void yz(int ki, int npts, int npk, int kjmin, float *out) const
    {
        for (int k = 0; k < npk; ++k)
            for (int j = 0; j < npts; ++j)
                nc_check(nc->read_f32(*v, 0, ((uint64_t)k * ny + (kjmin - 1 + j)) * nx + (ki - 1), 1, out + (size_t)k * npts + j), nc->err);
    }
};

static void file_example()
{
    printf("\n   EXAMPLE of dens_section.dat file\n   --------------------------------\n"
           "  Each section is described by 2 lines :\n"
           "    line#1 : name_of_section [variable_suffix] [ long_name_prefix ]\n"
           "    line#2 : imin  imax jmin jmax \n"
           "     IMPORTANT : the points indicated by imin,jmin  imax,jmax are F-point.\n"
           "  The list is closed by a line holding EOF.\n"
           "  example :\n03_Gibraltar gibra Gibraltar_Strait_transport_in_sigma_classes\n3378 3378 1956 1961\nEOF\n");
}

struct SectionData {   // what the reference holds for one section when the compute part starts (:559)
    int npts = 0, npk = 0, nk = 0;
    bool merid = false;
    std::vector<float> eu, de3, zu, zt, zs, zmask, rlonlat, ddepw;   // ddepw: -brk only
    std::vector<double> ddepu;                                       // (npk+1) x npts, row 0 = 0
};

// createvar attributes of one REAL(4) variable (cdfio.F90:371-459)
static int def_out_var(nc3::Writer &w, const std::string &name, const std::string &units, float fill, float vmin, float vmax,
                       const std::string &long_name, const std::string &short_name, int iweight, const std::string &axis,
                       const std::vector<int> &dims)
{
    const int id = w.def_var(name, nc3::NC_FLOAT, dims);
    w.put_att_text(id, "units", units);
    w.put_att_float(id, "_FillValue", fill);
    w.put_att_float(id, "valid_min", vmin);
    w.put_att_float(id, "valid_max", vmax);
    w.put_att_text(id, "long_name", long_name);
    w.put_att_text(id, "short_name", short_name);
    w.put_att_int(id, "iweight", iweight);
    w.put_att_text(id, "online_operation", "N/A");
    w.put_att_text(id, "axis", axis);
    w.put_att_float(id, "scale_factor", 1.f);
    w.put_att_float(id, "add_offset", 0.f);
    w.put_att_float(id, "savelog10", 0.f);
    return id;
}

int main(int argc, char **argv)
{
    Names cn;
    std::string cf_section = "dens_section.dat", cf_out = "trpsig.txt";
    if (argc == 1) {
        printf(" usage :  cdfsigtrp_gpu -t T-file -u U-file -v V-file [-s S-file] [-brk BRK-file] -smin sigma_min -smax sigma_max\n"
               "              -nbins nbins [-print] [-xtra] [-full] [-refdep ref_depth] [-neutral] [-section file] [-temp] [-help] [-teos10]\n"
               "     PURPOSE : density class transports across the zonal / meridional sections listed in %s (or along the\n"
               "               broken line of a BRK-file), computed on a B200 GPU.\n"
               "     REQUIRED FILES : %s, %s and %s (none of them with -brk)\n"
               "     OUTPUT : <section>_trpsig.nc (sigma_class, sigtrp in Sv) per section, and %s ;\n"
               "              -xtra: <section>_secdep.nc and <section>_secsig.nc ; -print: the tables on standard output\n"
               "     NOT IN THIS TWIN : -vvl, -full with -brk\n",
               cf_section.c_str(), cn.fhgr.c_str(), cn.fzgr.c_str(), cf_section.c_str(), cf_out.c_str());
        return 0;
    }
    std::string cf_tfil, cf_sfil = "none", cf_ufil, cf_vfil, cf_brk, cglobal;
    double dsigma_min = 0, dsigma_max = 0;
    int nbins = 0, ireq = 0, nreq = 6;
    float refdep = 0.f;
    bool lfull = false, lntr = false, ltemp = false, lteos10 = false, lbrk = false, lprint = false, lxtra = false;
    for (int i = 0; i < argc; ++i) cglobal += std::string(i ? " " : "") + argv[i];   // SetGlobalAtt: the command line
    for (int i = 1; i < argc;) {   // :228-256
        const std::string a = argv[i++];
        auto next = [&]() { return std::string(i < argc ? argv[i++] : ""); };
        if (a == "-t") { cf_tfil = next(); ++ireq; }
        else if (a == "-u") { cf_ufil = next(); ++ireq; }
        else if (a == "-v") { cf_vfil = next(); ++ireq; }
        else if (a == "-brk") { cf_brk = next(); ++ireq; lbrk = true; nreq = 4; }
        else if (a == "-smin") { dsigma_min = atof(next().c_str()); ++ireq; }
        else if (a == "-smax") { dsigma_max = atof(next().c_str()); ++ireq; }
        else if (a == "-nbins") { nbins = atoi(next().c_str()); ++ireq; }
        else if (a == "-s") { cf_sfil = next(); ++ireq; nreq = 7; }
        else if (a == "-full") lfull = true;
        else if (a == "-xtra") lxtra = true;
        else if (a == "-print") lprint = true;
        else if (a == "-temp") ltemp = true;
        else if (a == "-help") { file_example(); stop(99); }
        else if (a == "-refdep") refdep = (float)atof(next().c_str());
        else if (a == "-section") cf_section = next();
        else if (a == "-neutral") lntr = true;
        else if (a == "-teos10") lteos10 = true;
        else if (a == "-vvl") { printf(" ERROR : -vvl : not available in the GPU twin.\n"); stop(99); }
        else { printf(" ERROR : %s : unknown option.\n", a.c_str()); stop(99); }
    }
    if (cf_sfil == "none") cf_sfil = cf_tfil;
    if (ireq != nreq) { printf(" ERROR :  not enough input arguments. See the usage message and correct.\n"); stop(99); }
    if (nbins < 1) { printf(" ERROR : -nbins must be positive\n"); stop(99); }
    if (lbrk && lfull) { printf(" ERROR : -full with -brk : not available in the GPU twin.\n"); stop(99); }
    if (lbrk) {   // every file is the broken-line file (:268-276)
        cn.fzgr = cn.fhgr = cf_tfil = cf_sfil = cf_ufil = cf_vfil = cf_section = cf_brk;
    }
    bool lchk = chkfile(cn.fzgr);
    lchk = chkfile(cn.fhgr) || lchk; lchk = chkfile(cf_section) || lchk; lchk = chkfile(cf_tfil) || lchk;
    lchk = chkfile(cf_sfil) || lchk; lchk = chkfile(cf_ufil) || lchk; lchk = chkfile(cf_vfil) || lchk;
    if (lchk) stop(99);

    nc3::Reader ft, fs, fu, fv, hgr;
    nc_check(ft.open(cf_tfil), ft.err); nc_check(fs.open(cf_sfil), fs.err); nc_check(fu.open(cf_ufil), fu.err);
    nc_check(fv.open(cf_vfil), fv.err); nc_check(hgr.open(cn.fhgr), hgr.err);
    MeshZgr zgr;
    if (!lbrk) zgr.open(cn.fzgr);
    const Field T(ft, cn.votemper, cn), S(fs, cn.vosaline, cn), V(fv, cn.vomecrty, cn);
    std::unique_ptr<Field> U;
    if (!lbrk) U.reset(new Field(fu, "vozocrtx", cn));
    const float zsps = fs.spval(*S.v, cn.missing), zspu = lbrk ? 0.f : fu.spval(*U->v, cn.missing), zspv = fv.spval(*V.v, cn.missing);   // :289-291
    int iweight = 1;   // getatt(cf_vfil, cn_vomecrty, 'iweight'), 1 when absent (:314-315)
    if (const nc3::Att *a = V.v->att("iweight")) { iweight = (int)a->as_double(); if (iweight == 0) iweight = 1; }
    int mode = lntr ? 1 : 0;
    if (ltemp) {   // temperature decreases downward: change sign and swap the limits (:303-308)
        mode = 2;
        const double t = dsigma_max;
        dsigma_max = -dsigma_min;
        dsigma_min = -t;
    }
    std::vector<Section> sec;
    if (lbrk) {   // one pseudo-zonal section named after the file: <prefix>_<section>.nc (:329-343)
        Section s;
        s.imin = 1; s.imax = (int)ft.dim_len(cn.x, true); s.jmin = s.jmax = 1;
        const size_t u = cf_brk.rfind('_'), d = cf_brk.rfind('.');
        s.name = cf_brk.substr(u == std::string::npos ? 0 : u + 1, d == std::string::npos || d < u ? std::string::npos : d - (u == std::string::npos ? 0 : u + 1));
        s.varname = s.longname = s.name;
        sec.push_back(s);
    } else {
        sec = section_init(cf_section);
    }
    if (sec.empty()) { printf(" ERROR : no section in %s\n", cf_section.c_str()); stop(99); }
    const int npk = (int)ft.dim_len(cn.z, false);
    if (npk < 1) { printf(" ERROR : no vertical dimension %s in %s\n", cn.z.c_str(), cf_tfil.c_str()); stop(98); }
    std::vector<float> gdept(npk, 0.f), gdepw(npk, 0.f), e3t1d(npk), e3w1d(npk);
    if (!lbrk) {
        read_1d(zgr.nc, zgr.name1d("gdept"), npk, gdept.data());
        read_1d(zgr.nc, zgr.name1d("gdepw"), npk, gdepw.data());
    }
    if (lfull) {
        read_1d(zgr.nc, zgr.name1d("e3t1d"), npk, e3t1d.data());
        read_1d(zgr.nc, zgr.ver == "v2.0" ? "e3w" : zgr.ver == "v3.0" ? "e3w_0" : "e3w_1d", npk, e3w1d.data());   // getvare3 (cdfio.F90:2265-2274)
    }
    const std::string sfx = lbrk ? "" : zgr.ver == "v2.0" ? "_ps" : zgr.ver == "v3.0" ? "" : "_0";   // :418-422 / :510-514
    std::vector<double> tim(1, 0.0);
    { const int it = ft.find_var(cn.vtimec); if (it >= 0) ft.read_f64(ft.vars[it], 0, 0, 1, &tim[0]); }
    gpu_check(cdfgpu_init(-1, 1), "cdfgpu_init");

    std::vector<double> dsigma_lev(nbins + 1), dtrpbin((size_t)sec.size() * nbins, 0.0);
    {   // class limits (:355-359); the library returns the same values with every section
        const double dlt = (dsigma_max - dsigma_min) / nbins;
        for (int c = 0; c <= nbins; ++c) dsigma_lev[c] = dsigma_min + c * dlt;
    }
    for (size_t jsec = 0; jsec < sec.size(); ++jsec) {
        const Section &s = sec[jsec];
        SectionData q;
        q.npk = npk;
        if (s.imin == s.imax) { q.npts = s.jmax - s.jmin; q.merid = true; }
        else if (s.jmin == s.jmax) { q.npts = s.imax - s.imin; q.merid = false; }
        else {
            printf(" Section %s is neither zonal nor meridional :(\n We skip this section .\n", s.name.c_str());
            continue;
        }
        if (q.npts < 1) { printf(" Section %s is empty.\n We skip this section .\n", s.name.c_str()); continue; }
        const int npts = q.npts;
        const size_t n2 = (size_t)npts * npk;
        q.eu.resize(npts); q.de3.resize(n2); q.zu.resize(n2); q.zt.resize(n2); q.zs.resize(n2); q.zmask.resize(n2); q.rlonlat.resize(npts);
        q.ddepu.assign(n2 + npts, 0.0);
        q.nk = npk;   // (the reference leaves nk undefined when no level is all land, except with -brk)
        if (lbrk) {   // :465-495: everything comes from the broken-line file, columns imin .. imin+npts-1 of its single row
            Field(hgr, cn.e1v, cn).xz(s.jmin, npts, 1, s.imin, q.eu.data());
            Field(hgr, cn.vlon2d, cn).xz(s.jmin, npts, 1, s.imin, q.rlonlat.data());
            std::vector<float> t2(n2);
            q.ddepw.resize(n2);
            Field(ft, cn.ve3v, cn).xz(s.jmin, npts, npk, s.imin, q.de3.data());
            Field(ft, "depu3d", cn).xz(s.jmin, npts, npk, s.imin, t2.data());
            for (size_t c = 0; c < n2; ++c) q.ddepu[npts + c] = (double)t2[c];
            Field(ft, "depw3d", cn).xz(s.jmin, npts, npk, s.imin, q.ddepw.data());
            V.xz(s.jmin, npts, npk, s.imin, q.zu.data());
            T.xz(s.jmin, npts, npk, s.imin, q.zt.data());
            S.xz(s.jmin, npts, npk, s.imin, q.zs.data());
            Field(fv, cn.vmask, cn).xz(s.jmin, npts, npk, s.imin, q.zmask.data());
            for (auto &m : q.zmask) if (m == 9999.f) m = 0.f;   // fill value of the broken-line masks (:486)
            for (int k = 0; k < npk; ++k) {
                volatile float sum = 0.f;
                for (int i = 0; i < npts; ++i) sum = sum + q.zmask[(size_t)k * npts + i];
                if (sum == 0.f) { q.nk = k + 1; break; }
            }
        } else {
            std::vector<float> e3wa(n2), e3wb(n2), zsa(n2), zsb(n2), zta(n2), ztb(n2);
            std::unique_ptr<Field> e3w;   // (not read with -full)
            if (!lfull) e3w.reset(new Field(zgr.nc, "e3w" + sfx, cn));
            if (q.merid) {   // :404-460
                Field(hgr, "e2u", cn).yz(s.imin, npts, 1, s.jmin + 1, q.eu.data());
                Field(hgr, cn.vlat2d, cn).yz(s.imin, npts, 1, s.jmin + 1, q.rlonlat.data());
                if (!lfull) {
                    Field(zgr.nc, "e3u" + sfx, cn).yz(s.imin, npts, npk, s.jmin + 1, q.de3.data());
                    e3w->yz(s.imin, npts, npk, s.jmin + 1, e3wa.data());
                    e3w->yz(s.imin + 1, npts, npk, s.jmin + 1, e3wb.data());
                }
                U->yz(s.imin, npts, npk, s.jmin + 1, q.zu.data());
                S.yz(s.imin, npts, npk, s.jmin + 1, zsa.data());
                S.yz(s.imin + 1, npts, npk, s.jmin + 1, zsb.data());
                T.yz(s.imin, npts, npk, s.jmin + 1, zta.data());
                T.yz(s.imin + 1, npts, npk, s.jmin + 1, ztb.data());
            } else {         // :497-555
                Field(hgr, cn.e1v, cn).xz(s.jmin, npts, 1, s.imin, q.eu.data());   // (the reference starts e1v at imin, the data at imin+1)
                Field(hgr, cn.vlon2d, cn).xz(s.jmin, npts, 1, s.imin, q.rlonlat.data());
                if (!lfull) {
                    Field(zgr.nc, "e3v" + sfx, cn).xz(s.jmin, npts, npk, s.imin + 1, q.de3.data());
                    e3w->xz(s.jmin, npts, npk, s.imin + 1, e3wa.data());
                    e3w->xz(s.jmin + 1, npts, npk, s.imin + 1, e3wb.data());
                }
                V.xz(s.jmin, npts, npk, s.imin + 1, q.zu.data());
                S.xz(s.jmin, npts, npk, s.imin + 1, zsa.data());
                S.xz(s.jmin + 1, npts, npk, s.imin + 1, zsb.data());
                T.xz(s.jmin, npts, npk, s.imin + 1, zta.data());
                T.xz(s.jmin + 1, npts, npk, s.imin + 1, ztb.data());
            }
            if (lfull)
                for (int k = 0; k < npk; ++k)
                    for (int i = 0; i < npts; ++i) { q.de3[(size_t)k * npts + i] = e3t1d[k]; e3wa[(size_t)k * npts + i] = e3w1d[k]; e3wb[(size_t)k * npts + i] = e3w1d[k]; }
            // ---- the preparation of :428-460 / :521-555 (REAL(4) expressions, left to right)
            for (int i = 0; i < npts; ++i) q.ddepu[(size_t)npts + i] = (double)gdept[0];
            for (int k = 1; k < npk; ++k)
                for (int i = 0; i < npts; ++i) {
                    const size_t c = (size_t)k * npts + i;
                    const float m = e3wa[c] < e3wb[c] ? e3wa[c] : e3wb[c];
                    q.ddepu[c + npts] = q.ddepu[c] + (double)m;
                }
            const float zsp = q.merid ? zspu : zspv;
            for (size_t c = 0; c < n2; ++c) {
                if (q.zu[c] == zsp) q.zu[c] = 0.f;
                q.zmask[c] = (zsa[c] == zsps || zsb[c] == zsps) ? 0.f : 1.f;
                volatile float a = zsa[c] + zsb[c];
                a = 0.5f * a;
                q.zs[c] = a * q.zmask[c];
                volatile float t = zta[c] + ztb[c];
                t = 0.5f * t;
                q.zt[c] = q.merid ? t * q.zmask[c] : t;
            }
            for (int k = 0; k < npk; ++k) {
                volatile float sum = 0.f;
                for (int i = 0; i < npts; ++i) sum = sum + q.zs[(size_t)k * npts + i];
                if (sum == 0.f) { q.nk = k + 1; break; }
            }
            printf(q.merid ? "  NK =  %d\n" : " JMM nk   %d\n", q.nk);
        }
        const int nk = q.nk;
        const bool detail = lprint || lxtra;
        std::vector<double> dsig, dhiso, dwtrp, dwtrpbin;
        if (detail) { dsig.resize((size_t)(nk + 1) * npts); dhiso.resize((size_t)(nbins + 1) * npts); dwtrp.resize((size_t)(nbins + 1) * npts); dwtrpbin.resize((size_t)nbins * npts); }
        gpu_check(cdfsigtrp_gpu_section(npts, npk, nk, q.eu.data(), q.de3.data(), q.ddepu.data(), lbrk ? nullptr : gdepw.data(),
                                        lbrk ? q.ddepw.data() : nullptr, q.zu.data(), q.zt.data(), q.zs.data(), q.zmask.data(), mode,
                                        refdep, lteos10 ? 1 : 0, dsigma_min, dsigma_max, nbins, dsigma_lev.data(),
                                        detail ? dsig.data() : nullptr, detail ? dhiso.data() : nullptr, detail ? dwtrp.data() : nullptr,
                                        detail ? dwtrpbin.data() : nullptr, dtrpbin.data() + jsec * nbins),
                  "cdfsigtrp_gpu_section");
        const double *trp = dtrpbin.data() + jsec * nbins;
        if (lprint) {   // print_out (:902-963)
            auto table = [&](const char *title, int w0, int d0, int nrow, int d, auto label, auto value) {
                printf(" %s\n", title);
                for (int r = 0; r < nrow; ++r) {
                    if (d0 < 0) printf("%*d", w0, (int)label(r)); else printf("%s", fortran_f(label(r), w0, d0).c_str());
                    for (int i = 0; i < npts; ++i) printf("%s", fortran_f(value(i, r), 8, d).c_str());
                    printf("\n");
                }
            };
            auto lev = [&](int r) { return (double)(r + 1); };
            auto cls = [&](int r) { return dsigma_lev[r]; };
            table(" T (deg C)", 7, -1, nk, 3, lev, [&](int i, int k) { return (double)q.zt[(size_t)k * npts + i]; });
            table(" S (PSU)", 7, -1, nk, 3, lev, [&](int i, int k) { return (double)q.zs[(size_t)k * npts + i]; });
            table(" SIG (kg/m3 - 1000 )", 7, -1, nk, 3, lev, [&](int i, int k) { return dsig[(size_t)(k + 1) * npts + i]; });
            table(" VELOCITY (cm/s ) ", 7, -1, nk, 3, lev, [&](int i, int k) { return (double)(q.zu[(size_t)k * npts + i] * 100.f); });
            table(" GDEPU (m) ", 7, -1, nk, 0, lev, [&](int i, int k) { return q.ddepu[(size_t)(k + 1) * npts + i] * (double)q.zmask[(size_t)k * npts + i]; });
            table("E3 (m)", 7, -1, nk, 0, lev, [&](int i, int k) { return (double)q.de3[(size_t)k * npts + i] * (double)q.zmask[(size_t)k * npts + i]; });
            table(" DEP ISO ( m )", 7, 3, nbins + 1, 0, cls, [&](int i, int l) { return dhiso[(size_t)l * npts + i]; });
            table(" TRP SURF -->  ISO (SV)", 7, 3, nbins + 1, 3, cls, [&](int i, int l) { return dwtrp[(size_t)l * npts + i] / 1.e6; });
            printf("  TRP bins (SV)\n");
            for (int b = 0; b < nbins; ++b) {   // one value more than the format holds: it goes to a record of its own (format reversion)
                printf("%s", fortran_f(dsigma_lev[b], 7, 3).c_str());
                for (int i = 0; i < npts; ++i) printf("%s", fortran_f(dwtrpbin[(size_t)b * npts + i] / 1.e6, 8, 3).c_str());
                printf("\n%s\n", fortran_f(trp[b] / 1.e6, 7, 3).c_str());
            }
        }
        if (lxtra) {   // cdf_writ (:750-900): two (along section, depth | sigma) files
            const std::string sfxv = s.varname != "none" ? "_" + s.varname : "", pfx = s.longname != "none" ? s.longname + "_" : "";
            std::vector<float> row(npts);
            {
                nc3::Writer w;
                const int dx = w.def_dim("x", npts), dy = w.def_dim("y", 1), dz = w.def_dim("deptht", nk), dt = w.def_dim("time_counter", 0);
                const int vlon = w.def_var("nav_lon", nc3::NC_FLOAT, {dy, dx}), vlat = w.def_var("nav_lat", nc3::NC_FLOAT, {dy, dx});
                const int vz = w.def_var("deptht", nc3::NC_FLOAT, {dz});
                w.def_var("time_counter", nc3::NC_DOUBLE, {dt});
                const std::vector<int> d4 = {dt, dz, dy, dx};
                const int id[4] = {def_out_var(w, "temperature" + sfxv, "Celsius", 0.f, -2.f, 45.f, pfx + "Potential_temperature", "temperature", iweight, "XZT", d4),
                                   def_out_var(w, "salinity" + sfxv, "PSU", 0.f, 0.f, 45.f, pfx + "Salinity", "salinity", iweight, "XZT", d4),
                                   def_out_var(w, "density" + sfxv, "kg/m3 -1000", 0.f, 0.f, 45.f, pfx + "potential_density", "density", iweight, "XZT", d4),
                                   def_out_var(w, "velocity" + sfxv, "m/s", 0.f, -3.f, 3.f, pfx + "Normal_velocity", "velocity", iweight, "XZT", d4)};
                w.put_att_text(-1, "history", cglobal);
                nc_check(w.create(s.name + "_secdep.nc"), w.err);
                w.put_f32(vlon, 0, 0, npts, q.rlonlat.data());
                w.put_f32(vlat, 0, 0, npts, q.rlonlat.data());
                std::vector<float> dep(nk, 0.f);   // putheadervar copies the depth variable of the T file (cdfio.F90:2378-2398)
                for (const char *n : {"deptht", "depthu", "depthv", "depthw", "nav_lev", "z"})
                    if (ft.find_var(n) >= 0) { std::vector<float> all(npk); read_1d(ft, n, npk, all.data()); std::copy(all.begin(), all.begin() + nk, dep.begin()); break; }
                w.put_f32(vz, 0, 0, nk, dep.data());
                for (int k = 0; k < nk; ++k) {
                    nc_check(w.put_f32(id[0], 0, (uint64_t)k * npts, npts, q.zt.data() + (size_t)k * npts), w.err);
                    nc_check(w.put_f32(id[1], 0, (uint64_t)k * npts, npts, q.zs.data() + (size_t)k * npts), w.err);
                    for (int i = 0; i < npts; ++i) row[i] = (float)dsig[(size_t)(k + 1) * npts + i];
                    nc_check(w.put_f32(id[2], 0, (uint64_t)k * npts, npts, row.data()), w.err);
                    nc_check(w.put_f32(id[3], 0, (uint64_t)k * npts, npts, q.zu.data() + (size_t)k * npts), w.err);
                }
                w.close();
            }
            {
                nc3::Writer w;
                const int dx = w.def_dim("x", npts), dy = w.def_dim("y", 1), dz = w.def_dim("levels", nbins), dt = w.def_dim("time_counter", 0);
                const int vlon = w.def_var("nav_lon", nc3::NC_FLOAT, {dy, dx}), vlat = w.def_var("nav_lat", nc3::NC_FLOAT, {dy, dx});
                const int vz = w.def_var("levels", nc3::NC_FLOAT, {dz});
                w.def_var("time_counter", nc3::NC_DOUBLE, {dt});
                const std::vector<int> d4 = {dt, dz, dy, dx};
                const int id[3] = {def_out_var(w, "isodep" + sfxv, "m", 99999.f, 0.f, 6000.f, pfx + "isopycnal_depth", "isodep", iweight, "XST", d4),
                                   def_out_var(w, "bintrp" + sfxv, "SV", 99999.f, -5.f, 5.f, pfx + "Binned_transport", "bintrp", iweight, "XST", d4),
                                   def_out_var(w, "sumtrp" + sfxv, "SV", 99999.f, -20.f, 20.f, pfx + "cumulated_transport", "sumtrp", iweight, "XST", d4)};
                w.put_att_text(-1, "history", cglobal);
                nc_check(w.create(s.name + "_secsig.nc"), w.err);
                w.put_f32(vlon, 0, 0, npts, q.rlonlat.data());
                w.put_f32(vlat, 0, 0, npts, q.rlonlat.data());
                std::vector<float> l32(nbins);
                for (int b = 0; b < nbins; ++b) l32[b] = (float)dsigma_lev[b];
                w.put_f32(vz, 0, 0, nbins, l32.data());
                for (int b = 0; b < nbins; ++b) {   // isodep holds nbins-1 levels (ipk = nbins-1); the last level of the variable stays unwritten
                    if (b < nbins - 1) {
                        for (int i = 0; i < npts; ++i) row[i] = (float)dhiso[(size_t)b * npts + i];
                        nc_check(w.put_f32(id[0], 0, (uint64_t)b * npts, npts, row.data()), w.err);
                    }
                    for (int i = 0; i < npts; ++i) row[i] = (float)(dwtrpbin[(size_t)b * npts + i] / 1.e6);
                    nc_check(w.put_f32(id[1], 0, (uint64_t)b * npts, npts, row.data()), w.err);
                    for (int i = 0; i < npts; ++i) row[i] = (float)(dwtrp[(size_t)b * npts + i] / 1.e6);
                    nc_check(w.put_f32(id[2], 0, (uint64_t)b * npts, npts, row.data()), w.err);
                }
                w.close();
            }
        }
        double tot = 0.0;
        for (int b = 0; b < nbins; ++b) tot += trp[b];
        printf("  Total transport in all bins :%s %.10g\n", s.name.c_str(), tot / 1.e6);
    }

    // ---- trpsig.txt (:641-648): formats 9006, 9005, 9004 (:674-676)
    {
        FILE *f = fopen(cf_out.c_str(), "w");
        if (!f) { printf(" ERROR : cannot create %s\n", cf_out.c_str()); stop(99); }
        const size_t ipos = cf_tfil.find("_gridT.nc");
        fprintf(f, "# %s\n", ipos == std::string::npos ? "" : cf_tfil.substr(0, ipos).c_str());
        fprintf(f, "#%9s", " sigma  ");
        for (auto &s : sec) fprintf(f, "  %-12.12s  ", s.name.c_str());
        fprintf(f, "\n");
        for (int b = 0; b < nbins; ++b) {
            fprintf(f, "%9.4f", dsigma_lev[b]);
            for (size_t jsec = 0; jsec < sec.size(); ++jsec) fprintf(f, "%s", fortran_e16_7(dtrpbin[jsec * nbins + b]).c_str());
            fprintf(f, "\n");
        }
        fclose(f);
    }
    // ---- one file per section (CreateOutput, :965-1039; the values at :663-668)
    std::vector<float> lev32(nbins), trp32(nbins), zero(1, 0.f);
    for (int b = 0; b < nbins; ++b) lev32[b] = (float)dsigma_lev[b];
    for (size_t jsec = 0; jsec < sec.size(); ++jsec) {
        const Section &s = sec[jsec];
        const std::string sfxv = s.varname != "none" ? "_" + s.varname : "", pfx = s.longname != "none" ? s.longname + "_" : "";
        std::vector<OutVar> ov(2);
        if (ltemp) {
            ov[0] = {"temp_class", "class of potential temperature", "[]", 0.f, 100.f, 99999.f, "ZT"};
            ov[1] = {"temptrp" + sfxv, pfx + "transport in temperature class", "Sv", -1000.f, 1000.f, 99999.f, "ZT", "temptrp"};
        } else {
            ov[0] = {"sigma_class", "class of potential density", "[]", 0.f, 100.f, 99999.f, "ZT"};
            ov[1] = {"sigtrp" + sfxv, pfx + "transport in sigma class", "Sv", -1000.f, 1000.f, 99999.f, "ZT", "sigtrp"};
        }
        OutFile out;
        out.create(s.name + (ltemp ? "_trptemp.nc" : "_trpsig.nc"), "levels", 1, nbins, ov, cglobal, zero, lev32, tim, ft);
        for (int b = 0; b < nbins; ++b) trp32[b] = (float)(dtrpbin[jsec * nbins + b] / 1.e6);
        out.put(0, 0, lev32.data());
        out.put(1, 0, trp32.data());
        out.w.close();
    }
    gpu_check(cdfgpu_finalize(), "cdfgpu_finalize");
    return 0;
}
