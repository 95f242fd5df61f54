// Test helper (tests/test_packed_inputs.py): every value of one variable as the host reader delivers it
// (nc3::Reader::read_f32: int16 -> float, then the masked scale_factor and add_offset passes), written as raw float32 to
// <out>; on stdout, what nc3::Reader::packed_i16 reports for the variable.
#include <math.h>
#include <stdlib.h>

#include "../../cdftools_b200/csrc/host/nc3.hpp"

int main(int argc, char **argv)
{
    if (argc != 4) { fprintf(stderr, "usage: unpack_dump file.nc var out.bin\n"); return 2; }
    nc3::Reader r;
    if (!r.open(argv[1])) { fprintf(stderr, "%s\n", r.err.c_str()); return 1; }
    const int iv = r.find_var(argv[2]);
    if (iv < 0) { fprintf(stderr, "no variable %s\n", argv[2]); return 1; }
    const nc3::Var &v = r.vars[iv];
    const long nrec = v.isrec ? (long)r.numrecs : 1;
    std::vector<float> out((size_t)nrec * v.nelem_per_rec);
    for (long t = 0; t < nrec; ++t)
        if (!r.read_f32(v, t, 0, v.nelem_per_rec, out.data() + (size_t)t * v.nelem_per_rec)) { fprintf(stderr, "%s\n", r.err.c_str()); return 1; }
    FILE *f = fopen(argv[3], "wb");
    if (!f || fwrite(out.data(), sizeof(float), out.size(), f) != out.size()) return 1;
    fclose(f);
    float sf = 1.f, ao = 0.f, sp = 0.f;
    const bool packed = r.packed_i16(v, &sf, &ao, &sp);
    printf("{\"packed\": %s, \"sf\": %.9g, \"ao\": %.9g, \"sp\": %.9g}\n", packed ? "true" : "false", sf, ao, sp);
    return 0;
}
