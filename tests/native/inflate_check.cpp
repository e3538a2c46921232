// Host build of the device decoder's deflate core (bin3c_b200/csrc/inflate.cuh), for tests/test_bamdec_cpu.py, which
// compares it with zlib and builds it once more under AddressSanitizer + UBSan.
//   inflate_check inflate <raw deflate file> <out file> <capacity>   prints: <status> <bytes written>
//   inflate_check crc <file> <pieces>                                 prints: <crc> <crc of <pieces> parts combined>
// The second crc cuts the file into <pieces> parts of equal length (the last one shorter), takes each part's CRC on
// its own and joins them with crc32_combine, the way the device kernel joins the CRCs of a warp's 32 lanes.
#include <cinttypes>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../bin3c_b200/csrc/inflate.cuh"

static std::vector<uint8_t> slurp(const char *path) {
    std::vector<uint8_t> v;
    FILE *f = fopen(path, "rb");
    if (!f) exit(2);
    uint8_t buf[65536];
    size_t n;
    while ((n = fread(buf, 1, sizeof(buf), f)) > 0) v.insert(v.end(), buf, buf + n);
    fclose(f);
    return v;
}

int main(int argc, char **argv) {
    if (argc < 4) return 2;
    if (!strcmp(argv[1], "inflate") && argc == 5) {
        const std::vector<uint8_t> in = slurp(argv[2]);
        const int64_t cap = atoll(argv[4]);
        // exact-size buffers, so that ASan sees any read or write past either end
        uint8_t *src = (uint8_t *)malloc(in.size() ? in.size() : 1);
        if (!in.empty()) memcpy(src, in.data(), in.size());
        uint8_t *dst = (uint8_t *)malloc(cap ? cap : 1);
        int64_t n = 0;
        const int rc = b3c_inflate::inflate_raw(src, (int64_t)in.size(), dst, cap, &n);
        FILE *f = fopen(argv[3], "wb");
        if (!f) return 2;
        if (n) fwrite(dst, 1, n, f);
        fclose(f);
        free(src);
        free(dst);
        printf("%d %" PRId64 "\n", rc, n);
        return 0;
    }
    if (!strcmp(argv[1], "crc")) {
        const std::vector<uint8_t> in = slurp(argv[2]);
        const int64_t pieces = atoll(argv[3]), n = (int64_t)in.size();
        uint32_t table[256];
        b3c_inflate::crc32_table(table);
        const uint32_t whole = b3c_inflate::crc32_update(table, 0, in.data(), n);
        const int64_t len = pieces > 0 ? (n + pieces - 1) / pieces : n;
        uint32_t joined = 0;
        for (int64_t o = 0; o < n || o == 0; o += (len ? len : 1)) {
            const int64_t m = (o + len <= n) ? len : n - o;
            const uint32_t c = b3c_inflate::crc32_update(table, 0, in.data() + o, m);
            joined = o == 0 ? c : b3c_inflate::crc32_combine(joined, c, m);
            if (len == 0) break;
        }
        printf("%u %u\n", whole, joined);
        return 0;
    }
    return 2;
}
