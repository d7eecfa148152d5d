// Host build of the chunked deflate coder (csrc/deflate_core.h): the sequential definition of the bytes the device kernels
// write.  tests/test_deflate_cpu.py and tests/test_device_deflate.py drive it.
//   deflate_check streams IN OUT [IN OUT ...]     zlib stream of each raw input file
//   deflate_check lengths MAXBITS F0 F1 ...        Huffman code lengths for the given frequencies, one per line
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "../../adaptive-edge-aware-jpeg_b200/csrc/deflate_core.h"

static std::vector<uint8_t> slurp(const char* path) {
    std::vector<uint8_t> v;
    FILE* f = fopen(path, "rb");
    if (!f) { perror(path); exit(2); }
    uint8_t buf[1 << 16];
    size_t k;
    while ((k = fread(buf, 1, sizeof buf, f)) > 0) v.insert(v.end(), buf, buf + k);
    fclose(f);
    return v;
}

int main(int argc, char** argv) {
    if (argc >= 2 && !strcmp(argv[1], "streams")) {
        std::vector<uint16_t> prev(DF_CHUNK), head(1 << DF_HASH_BITS), tok(DF_CHUNK);
        DfWork w;
        for (int a = 2; a + 1 < argc; a += 2) {
            const std::vector<uint8_t> in = slurp(argv[a]);
            std::vector<uint8_t> out((size_t)df_stream_bound((int64_t)in.size()));
            const int64_t n = df_deflate_seq(in.data(), (int64_t)in.size(), out.data(), prev.data(), head.data(), tok.data(), &w);
            FILE* f = fopen(argv[a + 1], "wb");
            if (!f || fwrite(out.data(), 1, (size_t)n, f) != (size_t)n) { perror(argv[a + 1]); return 2; }
            fclose(f);
        }
        return 0;
    }
    if (argc >= 3 && !strcmp(argv[1], "lengths")) {
        const int maxbits = atoi(argv[2]), n = argc - 3;
        std::vector<uint32_t> freq(n), key(n), w(n);
        std::vector<uint8_t> lens(n);
        for (int i = 0; i < n; i++) freq[i] = (uint32_t)strtoul(argv[3 + i], nullptr, 10);
        df_huff_lengths(freq.data(), n, maxbits, lens.data(), key.data(), w.data());
        for (int i = 0; i < n; i++) printf("%d\n", lens[i]);
        return 0;
    }
    fprintf(stderr, "usage: deflate_check streams IN OUT ... | lengths MAXBITS F0 F1 ...\n");
    return 2;
}
