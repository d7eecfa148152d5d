// Host build of the segment-parallel zlib decoder (csrc/inflate_core.h): the sequential definition of what
// aeaj_inflate_coefficients gives.  tests/test_inflate_cpu.py and tests/test_device_inflate.py drive it.
//   inflate_check IN OUT
// IN: records of  u64 length, u64 expected output bytes, the zlib stream.
// OUT: per record  i32 status, i64 bytes produced, i32 merged segments, then the output if the status is 0.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "../../adaptive-edge-aware-jpeg_b200/csrc/inflate_core.h"

int main(int argc, char** argv) {
    if (argc != 3) { fprintf(stderr, "usage: inflate_check IN OUT\n"); return 2; }
    FILE* f = fopen(argv[1], "rb");
    FILE* g = fopen(argv[2], "wb");
    if (!f || !g) { perror("inflate_check"); return 2; }
    uint64_t hdr[2];
    while (fread(hdr, 8, 2, f) == 2) {
        std::vector<uint8_t> in(hdr[0] + 1), out(hdr[1] + 1);
        if (hdr[0] && fread(in.data(), 1, hdr[0], f) != hdr[0]) { fprintf(stderr, "short record\n"); return 2; }
        int64_t n = 0;
        int nseg = 0;
        const int32_t st = if_inflate_seq(in.data(), (int64_t)hdr[0], out.data(), (int64_t)hdr[1], (int64_t)hdr[1], &n, &nseg);
        const int32_t ns = nseg;
        fwrite(&st, 4, 1, g);
        fwrite(&n, 8, 1, g);
        fwrite(&ns, 4, 1, g);
        if (st == IF_OK) fwrite(out.data(), 1, (size_t)n, g);
    }
    fclose(f);
    return fclose(g) ? 2 : 0;
}
