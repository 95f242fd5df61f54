// nc3.hpp -- self-contained NetCDF classic (CDF-1 / CDF-2 "64-bit offset") reader and writer.
//
// libnetcdf does not exist in this image, so the host twins of cdfmoc / cdfmocsig carry their own I/O layer for the
// on-disk format the reference writes (src/cdfio.F90:295-298: NF90_64BIT_OFFSET) and that NEMO classic output uses.
// It plays the role of the cdfio routines on the hot path: getdim (cdfio.F90:876-1003), getvar (:1425-1609),
// getvar1d (:2151-2186), getvare3 (:2189-2287), getspval (:1006-1039), create/createvar/putatt/putheadervar/putvar
// (:260-459, :629-682, :2290-2407, :2642-2681).  NetCDF-4/HDF5 files are out of reach here (documented limitation).
//
// A record can be fetched as RAW big-endian bytes straight into a pinned buffer (read_raw) -- the byte swap then
// happens on the GPU (K3, cdfgpu_set_input_big_endian; for NC_SHORT the unpacking too, K3b) -- or converted on the
// host (read_f32).
#pragma once
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <unistd.h>

#include <algorithm>
#include <string>
#include <thread>
#include <vector>

namespace nc3 {

enum { NC_BYTE = 1, NC_CHAR = 2, NC_SHORT = 3, NC_INT = 4, NC_FLOAT = 5, NC_DOUBLE = 6 };
enum { TAG_DIM = 0x0A, TAG_VAR = 0x0B, TAG_ATT = 0x0C };

inline size_t type_size(int t) { return t == NC_BYTE || t == NC_CHAR ? 1 : t == NC_SHORT ? 2 : t == NC_DOUBLE ? 8 : 4; }
inline uint32_t bswap32(uint32_t v) { return __builtin_bswap32(v); }
inline uint64_t bswap64(uint64_t v) { return __builtin_bswap64(v); }
inline size_t pad4(size_t n) { return (n + 3) & ~(size_t)3; }

struct Att {
    std::string name;
    int type = 0;
    size_t nelems = 0;
    std::vector<unsigned char> data;  // native-endian values
    double as_double(size_t i = 0) const
    {
        if (i >= nelems) return 0.0;
        switch (type) {
        case NC_BYTE: return (double)((const signed char *)data.data())[i];
        case NC_SHORT: return (double)((const int16_t *)data.data())[i];
        case NC_INT: return (double)((const int32_t *)data.data())[i];
        case NC_FLOAT: return (double)((const float *)data.data())[i];
        case NC_DOUBLE: return ((const double *)data.data())[i];
        }
        return 0.0;
    }
    std::string as_string() const { return std::string((const char *)data.data(), type == NC_CHAR ? nelems : 0); }
};
struct Dim {
    std::string name;
    uint64_t len = 0;
};
struct Var {
    std::string name;
    int type = 0;
    std::vector<int> dimids;
    std::vector<Att> atts;
    uint64_t vsize = 0, begin = 0;
    bool isrec = false;
    uint64_t nelem_per_rec = 0;  // elements of one record (record vars) or of the whole variable
    const Att *att(const std::string &n) const
    {
        for (auto &a : atts)
            if (a.name == n) return &a;
        return nullptr;
    }
};

inline void swap_range(void *p, size_t n, size_t es)
{
    if (es == 2) { uint16_t *q = (uint16_t *)p; for (size_t i = 0; i < n; ++i) q[i] = __builtin_bswap16(q[i]); }
    else if (es == 4) { uint32_t *q = (uint32_t *)p; for (size_t i = 0; i < n; ++i) q[i] = bswap32(q[i]); }
    else if (es == 8) { uint64_t *q = (uint64_t *)p; for (size_t i = 0; i < n; ++i) q[i] = bswap64(q[i]); }
}
// threads for the bulk work of the host reader (positional reads of whole records, byte swaps of the mesh fields):
// $CDFGPU_READ_THREADS, else the hardware's concurrency, at most 16
inline int io_threads()
{
    static int n = 0;
    if (n == 0) {
        const char *e = getenv("CDFGPU_READ_THREADS");
        n = e && atoi(e) > 0 ? atoi(e) : (int)std::thread::hardware_concurrency();
        n = n < 1 ? 1 : n > 16 ? 16 : n;
    }
    return n;
}
inline void swap_inplace(void *p, size_t n, size_t es)
{
    const int nt = io_threads();
    if (es == 1) return;
    if (n < ((size_t)1 << 22) || nt == 1) { swap_range(p, n, es); return; }
    std::vector<std::thread> th;
    const size_t chunk = (n + nt - 1) / nt;
    for (int t = 0; t < nt; ++t) {
        const size_t a = (size_t)t * chunk, b = a + chunk < n ? a + chunk : n;
        if (a < b) th.emplace_back([=]() { swap_range((char *)p + a * es, b - a, es); });
    }
    for (auto &x : th) x.join();
}

class Reader {
  public:
    int version = 0;
    uint64_t numrecs = 0, recsize = 0;
    int recdim = -1;
    std::vector<Dim> dims;
    std::vector<Att> gatts;
    std::vector<Var> vars;
    std::string path, err;

    ~Reader() { close(); }
    void close() { if (f_) fclose(f_); f_ = nullptr; }

    bool open(const std::string &p)
    {
        path = p;
        f_ = fopen(p.c_str(), "rb");
        if (!f_) { err = "cannot open " + p; return false; }
        unsigned char magic[4];
        if (fread(magic, 1, 4, f_) != 4 || magic[0] != 'C' || magic[1] != 'D' || magic[2] != 'F') {
            err = p + ": not a NetCDF classic file (NetCDF-4/HDF5 is not supported by this reader)";
            return false;
        }
        version = magic[3];
        if (version != 1 && version != 2) { err = p + ": unsupported CDF version"; return false; }
        uint32_t nr = 0;
        if (!rd32(nr)) return fail();
        if (!read_dims() || !read_atts(gatts) || !read_vars()) return fail();
        // record size and element counts
        recsize = 0;
        int nrecvars = 0;
        for (auto &v : vars) {
            uint64_t n = 1;
            for (size_t d = 0; d < v.dimids.size(); ++d)
                if (!(d == 0 && v.isrec)) n *= dims[v.dimids[d]].len;
            v.nelem_per_rec = n;
            if (v.isrec) { recsize += v.vsize; ++nrecvars; }
        }
        if (nrecvars == 1)  // a single record variable is not padded
            for (auto &v : vars)
                if (v.isrec) recsize = v.nelem_per_rec * type_size(v.type);
        numrecs = nr;
        if (nr == 0xFFFFFFFFu && recsize) {  // streaming: derive from the file size
            uint64_t first = ~0ull;
            for (auto &v : vars) if (v.isrec && v.begin < first) first = v.begin;
            fseeko(f_, 0, SEEK_END);
            numrecs = ((uint64_t)ftello(f_) - first) / recsize;
        }
        if (recdim >= 0) dims[recdim].len = numrecs;
        return true;
    }

    int find_var(const std::string &n) const
    {
        for (size_t i = 0; i < vars.size(); ++i)
            if (vars[i].name == n) return (int)i;
        return -1;
    }
    // getdim (cdfio.F90:876-1003): cn_x is matched exactly, the others by substring
    long dim_len(const std::string &pattern, bool exact) const
    {
        for (auto &d : dims)
            if (exact ? d.name == pattern : d.name.find(pattern) != std::string::npos) return (long)d.len;
        return 0;
    }
    // getspval (cdfio.F90:1006-1039)
    float spval(const Var &v, const std::string &cn_missing = "_FillValue") const
    {
        const char *tries[] = {cn_missing.c_str(), "missing_value", "Fillvalue", "_Fillvalue"};
        for (auto t : tries)
            if (const Att *a = v.att(t)) return (float)a->as_double();
        return 0.f;
    }
    uint64_t offset_of(const Var &v, long rec, uint64_t elem_off) const
    {
        return v.begin + (v.isrec ? (uint64_t)rec * recsize : 0) + elem_off * type_size(v.type);
    }
    // raw big-endian bytes of `nelem` elements starting at element `elem_off` of record `rec`
    bool read_raw(const Var &v, long rec, uint64_t elem_off, uint64_t nelem, void *out)
    {
        const off_t off = (off_t)offset_of(v, rec, elem_off);
        const size_t nb = nelem * type_size(v.type);
        if (nb >= ((size_t)64 << 20)) {   // a whole 3-D record: positional reads from several threads (one memcpy stream
                                          // out of the page cache tops out near 3 GB/s, well below PCIe)
            const int fd = fileno(f_);
            const int nt = io_threads();
            const size_t chunk = ((nb + nt - 1) / nt + 4095) & ~(size_t)4095;
            std::vector<std::thread> th;
            std::vector<int> ok(nt, 1);
            for (int t = 0; t < nt; ++t)
                th.emplace_back([&, t]() {
                    size_t b0 = (size_t)t * chunk, b1 = b0 + chunk < nb ? b0 + chunk : nb;
                    while (b0 < b1) {
                        const ssize_t r = pread(fd, (char *)out + b0, b1 - b0, off + (off_t)b0);
                        if (r <= 0) { ok[t] = 0; return; }
                        b0 += (size_t)r;
                    }
                });
            for (auto &x : th) x.join();
            for (int t = 0; t < nt; ++t)
                if (!ok[t]) { err = "short read of " + v.name + " in " + path; return false; }
            return true;
        }
        if (fseeko(f_, off, SEEK_SET)) { err = "seek failed in " + path; return false; }
        if (fread(out, 1, nb, f_) != nb) { err = "short read of " + v.name + " in " + path; return false; }
        return true;
    }
    // values converted to float, with scale_factor / add_offset / savelog10 applied as getvar does (cdfio.F90:1563-1605)
    bool read_f32(const Var &v, long rec, uint64_t elem_off, uint64_t nelem, float *out)
    {
        const size_t es = type_size(v.type);
        std::vector<unsigned char> tmp;
        void *buf = out;
        if (v.type != NC_FLOAT) { tmp.resize(nelem * es); buf = tmp.data(); }
        if (!read_raw(v, rec, elem_off, nelem, buf)) return false;
        swap_inplace(buf, nelem, es);
        switch (v.type) {
        case NC_FLOAT: break;
        case NC_BYTE: for (uint64_t i = 0; i < nelem; ++i) out[i] = (float)((signed char *)buf)[i]; break;
        case NC_SHORT: for (uint64_t i = 0; i < nelem; ++i) out[i] = (float)((int16_t *)buf)[i]; break;
        case NC_INT: for (uint64_t i = 0; i < nelem; ++i) out[i] = (float)((int32_t *)buf)[i]; break;
        case NC_DOUBLE: for (uint64_t i = 0; i < nelem; ++i) out[i] = (float)((double *)buf)[i]; break;
        default: err = v.name + ": not a numeric variable"; return false;
        }
        // Caution : order does matter (cdfio.F90:1599-1602): three separate passes, each one skipping the values that equal
        // the missing value AT THAT POINT -- scaled values are compared again before the offset is added
        float sf = 1.f, ao = 0.f;
        needs_unpack(v, &sf, &ao);
        const float sp = spval(v);
        if (sf != 1.f)
            for (uint64_t i = 0; i < nelem; ++i) if (out[i] != sp) out[i] = out[i] * sf;
        if (ao != 0.f)
            for (uint64_t i = 0; i < nelem; ++i) if (out[i] != sp) { volatile float t = out[i] + ao; out[i] = t; }
        if (has_log(v))
            for (uint64_t i = 0; i < nelem; ++i) if (out[i] != sp) out[i] = __builtin_powf(10.f, out[i]);
        return true;
    }
    bool read_f64(const Var &v, long rec, uint64_t elem_off, uint64_t nelem, double *out)
    {
        if (v.type == NC_DOUBLE) {
            if (!read_raw(v, rec, elem_off, nelem, out)) return false;
            swap_inplace(out, nelem, 8);
            return true;
        }
        std::vector<float> t(nelem);
        if (!read_f32(v, rec, elem_off, nelem, t.data())) return false;
        for (uint64_t i = 0; i < nelem; ++i) out[i] = t[i];
        return true;
    }
    // true when the variable is stored as plain float32 with no packing: eligible for the raw + GPU byte-swap path
    bool is_plain_f32(const Var &v) const { return v.type == NC_FLOAT && !needs_unpack(v, nullptr, nullptr) && !has_log(v); }
    // true when the variable is NC_SHORT without savelog10: its raw 16-bit values can be unpacked on the GPU (K3b,
    // cdfgpu_set_input_packing) with the scale_factor, add_offset and missing value read_f32 would use
    bool packed_i16(const Var &v, float *sf, float *ao, float *sp) const
    {
        if (v.type != NC_SHORT || has_log(v)) return false;
        needs_unpack(v, sf, ao);
        *sp = spval(v);
        return true;
    }

  private:
    FILE *f_ = nullptr;
    bool fail() { if (err.empty()) err = path + ": truncated or corrupt header"; return false; }
    bool has_log(const Var &v) const { const Att *a = v.att("savelog10"); return a && a->as_double() != 0.0; }
    bool needs_unpack(const Var &v, float *sf, float *ao) const
    {
        float s = 1.f, o = 0.f;
        if (const Att *a = v.att("scale_factor")) s = (float)a->as_double();
        if (const Att *a = v.att("add_offset")) o = (float)a->as_double();
        if (sf) *sf = s;
        if (ao) *ao = o;
        return s != 1.f || o != 0.f;
    }
    bool rd32(uint32_t &v) { if (fread(&v, 4, 1, f_) != 1) return false; v = bswap32(v); return true; }
    bool rd64(uint64_t &v) { if (fread(&v, 8, 1, f_) != 1) return false; v = bswap64(v); return true; }
    bool rdname(std::string &s)
    {
        uint32_t n;
        if (!rd32(n) || n > (1u << 20)) return false;
        std::vector<char> b(pad4(n));
        if (n && fread(b.data(), 1, b.size(), f_) != b.size()) return false;
        s.assign(b.data(), n);
        return true;
    }
    bool read_dims()
    {
        uint32_t tag, n;
        if (!rd32(tag) || !rd32(n)) return false;
        if (tag == 0 && n == 0) return true;
        if (tag != TAG_DIM) return false;
        dims.resize(n);
        for (uint32_t i = 0; i < n; ++i) {
            uint32_t len;
            if (!rdname(dims[i].name) || !rd32(len)) return false;
            dims[i].len = len;
            if (len == 0) recdim = (int)i;
        }
        return true;
    }
    bool read_atts(std::vector<Att> &atts)
    {
        uint32_t tag, n;
        if (!rd32(tag) || !rd32(n)) return false;
        if (tag == 0 && n == 0) return true;
        if (tag != TAG_ATT) return false;
        atts.resize(n);
        for (uint32_t i = 0; i < n; ++i) {
            uint32_t ty, ne;
            if (!rdname(atts[i].name) || !rd32(ty) || !rd32(ne)) return false;
            atts[i].type = (int)ty;
            atts[i].nelems = ne;
            const size_t nb = (size_t)ne * type_size((int)ty);
            atts[i].data.resize(pad4(nb) + 8);
            if (nb && fread(atts[i].data.data(), 1, pad4(nb), f_) != pad4(nb)) return false;
            swap_inplace(atts[i].data.data(), ne, type_size((int)ty));
        }
        return true;
    }
    bool read_vars()
    {
        uint32_t tag, n;
        if (!rd32(tag) || !rd32(n)) return false;
        if (tag == 0 && n == 0) return true;
        if (tag != TAG_VAR) return false;
        vars.resize(n);
        for (uint32_t i = 0; i < n; ++i) {
            Var &v = vars[i];
            uint32_t nd, ty, vs;
            if (!rdname(v.name) || !rd32(nd)) return false;
            v.dimids.resize(nd);
            for (uint32_t d = 0; d < nd; ++d) {
                uint32_t id;
                if (!rd32(id) || id >= dims.size()) return false;
                v.dimids[d] = (int)id;
            }
            if (!read_atts(v.atts) || !rd32(ty) || !rd32(vs)) return false;
            v.type = (int)ty;
            v.vsize = vs;
            if (version == 1) { uint32_t b; if (!rd32(b)) return false; v.begin = b; }
            else if (!rd64(v.begin)) return false;
            v.isrec = nd > 0 && v.dimids[0] == recdim;
        }
        return true;
    }
};

// ---- writer: CDF-2, one unlimited dimension, everything defined before the first write --------------------------------
class Writer {
  public:
    std::string err;
    ~Writer() { close(); }
    int def_dim(const std::string &name, uint64_t len)  // len 0 = unlimited
    {
        Dim d; d.name = name; d.len = len;
        dims_.push_back(d);
        if (len == 0) recdim_ = (int)dims_.size() - 1;
        return (int)dims_.size() - 1;
    }
    int def_var(const std::string &name, int type, const std::vector<int> &dimids)
    {
        Var v; v.name = name; v.type = type; v.dimids = dimids;
        v.isrec = !dimids.empty() && dimids[0] == recdim_;
        vars_.push_back(v);
        return (int)vars_.size() - 1;
    }
    void put_att_text(int varid, const std::string &name, const std::string &val)
    {
        Att a; a.name = name; a.type = NC_CHAR; a.nelems = val.size();
        a.data.assign(val.begin(), val.end());
        (varid < 0 ? gatts_ : vars_[varid].atts).push_back(a);
    }
    void put_att_float(int varid, const std::string &name, float val)
    {
        Att a; a.name = name; a.type = NC_FLOAT; a.nelems = 1; a.data.resize(4);
        memcpy(a.data.data(), &val, 4);
        (varid < 0 ? gatts_ : vars_[varid].atts).push_back(a);
    }
    void put_att_int(int varid, const std::string &name, int32_t val)
    {
        Att a; a.name = name; a.type = NC_INT; a.nelems = 1; a.data.resize(4);
        memcpy(a.data.data(), &val, 4);
        (varid < 0 ? gatts_ : vars_[varid].atts).push_back(a);
    }
    bool create(const std::string &path)
    {
        f_ = fopen(path.c_str(), "wb+");
        if (!f_) { err = "cannot create " + path; return false; }
        // layout: fixed variables first, then the record variables
        std::vector<unsigned char> hdr;
        build_header(hdr, 0);             // first pass for the size (begins are fixed-width in CDF-2)
        uint64_t pos = pad4(hdr.size());
        for (auto &v : vars_) if (!v.isrec) { set_sizes(v); v.begin = pos; pos += v.vsize; }
        recbegin_ = pos;
        recsize_ = 0;
        for (auto &v : vars_) if (v.isrec) { set_sizes(v); v.begin = pos; pos += v.vsize; recsize_ += v.vsize; }
        hdr.clear();
        build_header(hdr, 0);
        hdr.resize(pad4(hdr.size()), 0);
        if (fwrite(hdr.data(), 1, hdr.size(), f_) != hdr.size()) { err = "write failed"; return false; }
        // pre-extend the fixed part
        if (recbegin_ > hdr.size()) {
            std::vector<unsigned char> z(recbegin_ - hdr.size(), 0);
            fwrite(z.data(), 1, z.size(), f_);
        }
        return true;
    }
    // nelem values starting at element elem_off of record rec (ignored for fixed variables); host-endian input
    bool put_f32(int varid, long rec, uint64_t elem_off, uint64_t nelem, const float *vals)
    {
        std::vector<uint32_t> t(nelem);
        for (uint64_t i = 0; i < nelem; ++i) { uint32_t u; memcpy(&u, vals + i, 4); t[i] = bswap32(u); }
        return put_bytes(varid, rec, elem_off * 4, t.data(), nelem * 4);
    }
    bool put_f64(int varid, long rec, uint64_t elem_off, uint64_t nelem, const double *vals)
    {
        std::vector<uint64_t> t(nelem);
        for (uint64_t i = 0; i < nelem; ++i) { uint64_t u; memcpy(&u, vals + i, 8); t[i] = bswap64(u); }
        return put_bytes(varid, rec, elem_off * 8, t.data(), nelem * 8);
    }
    void close()
    {
        if (!f_) return;
        // pad the last record to the record size and patch numrecs
        if (numrecs_ && recsize_) {
            fseeko(f_, 0, SEEK_END);
            const uint64_t want = recbegin_ + numrecs_ * recsize_;
            uint64_t have = (uint64_t)ftello(f_);
            if (have < want) { std::vector<unsigned char> z(want - have, 0); fwrite(z.data(), 1, z.size(), f_); }
        }
        uint32_t nr = bswap32((uint32_t)numrecs_);
        fseeko(f_, 4, SEEK_SET);
        fwrite(&nr, 4, 1, f_);
        fclose(f_);
        f_ = nullptr;
    }

  private:
    FILE *f_ = nullptr;
    std::vector<Dim> dims_;
    std::vector<Att> gatts_;
    std::vector<Var> vars_;
    int recdim_ = -1;
    uint64_t recbegin_ = 0, recsize_ = 0, numrecs_ = 0;

    void set_sizes(Var &v)
    {
        uint64_t n = 1;
        for (size_t d = 0; d < v.dimids.size(); ++d)
            if (!(d == 0 && v.isrec)) n *= dims_[v.dimids[d]].len;
        v.nelem_per_rec = n;
        v.vsize = pad4(n * type_size(v.type));
    }
    bool put_bytes(int varid, long rec, uint64_t byte_off, const void *p, size_t nb)
    {
        const Var &v = vars_[varid];
        const uint64_t off = v.begin + (v.isrec ? (uint64_t)rec * recsize_ : 0) + byte_off;
        if (fseeko(f_, (off_t)off, SEEK_SET) || fwrite(p, 1, nb, f_) != nb) { err = "write failed"; return false; }
        if (v.isrec && (uint64_t)rec + 1 > numrecs_) numrecs_ = (uint64_t)rec + 1;
        return true;
    }
    static void w32(std::vector<unsigned char> &b, uint32_t v) { v = bswap32(v); b.insert(b.end(), (unsigned char *)&v, (unsigned char *)&v + 4); }
    static void w64(std::vector<unsigned char> &b, uint64_t v) { v = bswap64(v); b.insert(b.end(), (unsigned char *)&v, (unsigned char *)&v + 8); }
    static void wname(std::vector<unsigned char> &b, const std::string &s)
    {
        w32(b, (uint32_t)s.size());
        b.insert(b.end(), s.begin(), s.end());
        b.resize(pad4(b.size()), 0);
    }
    static void watts(std::vector<unsigned char> &b, const std::vector<Att> &atts)
    {
        if (atts.empty()) { w32(b, 0); w32(b, 0); return; }
        w32(b, TAG_ATT); w32(b, (uint32_t)atts.size());
        for (auto &a : atts) {
            wname(b, a.name);
            w32(b, (uint32_t)a.type); w32(b, (uint32_t)a.nelems);
            std::vector<unsigned char> d(a.data.begin(), a.data.begin() + a.nelems * type_size(a.type));
            swap_inplace(d.data(), a.nelems, type_size(a.type));
            b.insert(b.end(), d.begin(), d.end());
            b.resize(pad4(b.size()), 0);
        }
    }
    void build_header(std::vector<unsigned char> &b, uint32_t numrecs)
    {
        b.push_back('C'); b.push_back('D'); b.push_back('F'); b.push_back(2);
        w32(b, numrecs);
        w32(b, TAG_DIM); w32(b, (uint32_t)dims_.size());
        for (auto &d : dims_) { wname(b, d.name); w32(b, (uint32_t)d.len); }
        watts(b, gatts_);
        w32(b, TAG_VAR); w32(b, (uint32_t)vars_.size());
        for (auto &v : vars_) {
            wname(b, v.name);
            w32(b, (uint32_t)v.dimids.size());
            for (int id : v.dimids) w32(b, (uint32_t)id);
            watts(b, v.atts);
            w32(b, (uint32_t)v.type);
            w32(b, (uint32_t)std::min<uint64_t>(v.vsize, 0xFFFFFFFFu));
            w64(b, v.begin);
        }
    }
};

}  // namespace nc3
