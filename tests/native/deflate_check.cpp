// Host build of the device encoder's deflate core (bin3c_b200/csrc/deflate.cuh), for tests/test_bgzf_deflate_cpu.py,
// which compares it with zlib and builds it once more under AddressSanitizer + UBSan.
//   deflate_check lengths <limit> <freq>...   prints the code lengths huff_lengths gives the frequencies
//   deflate_check <in file> <out file>
// cuts the input into members of MEMBER_INPUT bytes, writes the members one after the other (no end-of-file member)
// and checks each one against its own input: BGZF header and BSIZE, the payload inflated by inflate.cuh's host build,
// CRC-32 and ISIZE, and for a dynamic block the code lengths read back from its header (within 15 / 7 bits, every code
// complete).  Prints one line per member:  <index> <block type> <member bytes> <max lit/len bits> <max dist bits>
// <max code-length bits> <status>, status 0 when every check passed.
#include <cinttypes>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <vector>

#include "../../bin3c_b200/csrc/deflate.cuh"

namespace D = b3c_deflate;
namespace I = b3c_inflate;

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

static uint32_t rd32(const uint8_t *p) { return p[0] | (p[1] << 8) | (p[2] << 16) | ((uint32_t)p[3] << 24); }

// sum of 2^-len over the codes, scaled by 2^15: 32768 for a complete code
static int64_t kraft(const uint8_t *len, int n) {
    int64_t k = 0;
    for (int s = 0; s < n; ++s)
        if (len[s]) k += (int64_t)1 << (15 - len[s]);
    return k;
}

// reads the code lengths of the dynamic block header at p; returns false on a malformed header
static bool header_lengths(const uint8_t *p, int64_t n, int *max_l, int *max_d, int *max_c) {
    I::State s;
    memset(&s, 0, sizeof(s));
    s.in = p;
    s.in_len = n;
    I::bits(s, 3);
    const int nlen = (int)I::bits(s, 5) + 257, ndist = (int)I::bits(s, 5) + 1, ncode = (int)I::bits(s, 4) + 4;
    const uint8_t ORDER[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    uint8_t cl[19] = {0}, lengths[D::MAX_RLE] = {0};
    for (int k = 0; k < ncode; ++k) cl[ORDER[k]] = (uint8_t)I::bits(s, 3);
    *max_c = 0;
    for (int k = 0; k < 19; ++k) *max_c = cl[k] > *max_c ? cl[k] : *max_c;
    I::Huffman h;
    if (I::construct(h, cl, 19) != 0 || kraft(cl, 19) != 32768) return false;
    for (int idx = 0; idx < nlen + ndist;) {
        const int sym = I::decode(s, h);
        if (sym < 0) return false;
        if (sym < 16) {
            lengths[idx++] = (uint8_t)sym;
            continue;
        }
        int rep, v = 0;
        if (sym == 16) {
            if (idx == 0) return false;
            v = lengths[idx - 1];
            rep = 3 + (int)I::bits(s, 2);
        } else {
            rep = sym == 17 ? 3 + (int)I::bits(s, 3) : 11 + (int)I::bits(s, 7);
        }
        if (idx + rep > nlen + ndist) return false;
        while (rep--) lengths[idx++] = (uint8_t)v;
    }
    *max_l = *max_d = 0;
    for (int k = 0; k < nlen; ++k) *max_l = lengths[k] > *max_l ? lengths[k] : *max_l;
    for (int k = 0; k < ndist; ++k) *max_d = lengths[nlen + k] > *max_d ? lengths[nlen + k] : *max_d;
    return !s.overrun && lengths[256] != 0 && kraft(lengths, nlen) == 32768 && kraft(lengths + nlen, ndist) == 32768;
}

int main(int argc, char **argv) {
    if (argc >= 3 && !strcmp(argv[1], "lengths")) {
        const int limit = atoi(argv[2]), n = argc - 3;
        if (n < 2 || n > D::LCODES) return 2;
        uint32_t freq[D::LCODES];
        uint8_t len[D::LCODES];
        for (int s = 0; s < n; ++s) freq[s] = (uint32_t)strtoul(argv[3 + s], nullptr, 10);
        D::huff_lengths(freq, n, limit, len);
        for (int s = 0; s < n; ++s) printf("%d%c", len[s], s + 1 < n ? ' ' : '\n');
        return 0;
    }
    if (argc != 3) return 2;
    const std::vector<uint8_t> in = slurp(argv[1]);
    FILE *f = fopen(argv[2], "wb");
    if (!f) return 2;
    std::unique_ptr<D::Scratch> S(new D::Scratch);
    uint32_t table[256];
    I::crc32_table(table);
    const int64_t n_all = (int64_t)in.size();
    for (int64_t lo = 0, idx = 0; lo < n_all || (n_all == 0 && idx == 0); lo += D::MEMBER_INPUT, ++idx) {
        const int n = (int)(n_all - lo < D::MEMBER_INPUT ? n_all - lo : D::MEMBER_INPUT);
        // exact-size buffers, so that ASan sees any read or write past either end
        uint8_t *src = (uint8_t *)malloc(n ? n : 1);
        if (n) memcpy(src, in.data() + lo, n);
        uint8_t *m = (uint8_t *)malloc(D::MEMBER_MAX);
        const int bytes = D::deflate_member(src, n, m, *S);
        fwrite(m, 1, bytes, f);
        int status = 0, max_l = 0, max_d = 0, max_c = 0;
        const uint8_t head[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
        const int64_t plen = bytes - D::HEADER_BYTES - D::TRAILER_BYTES;
        const int btype = (m[D::HEADER_BYTES] >> 1) & 3;
        if (bytes > D::MEMBER_MAX || memcmp(m, head, 16) != 0 || m[16] + (m[17] << 8) != bytes - 1) status = 1;
        uint8_t *back = (uint8_t *)malloc(n ? n : 1);
        int64_t got = 0;
        if (I::inflate_raw(m + D::HEADER_BYTES, plen, back, n, &got) != I::OK || got != n ||
            (n && memcmp(back, src, n) != 0))
            status = status ? status : 2;
        if (rd32(m + bytes - 8) != I::crc32_update(table, 0, src, n) || rd32(m + bytes - 4) != (uint32_t)n)
            status = status ? status : 3;
        if (btype == 2 && !header_lengths(m + D::HEADER_BYTES, plen, &max_l, &max_d, &max_c)) status = status ? status : 4;
        if (btype == 2 && (max_l > 15 || max_d > 15 || max_c > 7)) status = status ? status : 5;
        if (btype != 0 && btype != 2) status = status ? status : 6;
        printf("%" PRId64 " %d %d %d %d %d %d\n", idx, btype, bytes, max_l, max_d, max_c, status);
        free(back);
        free(src);
        free(m);
    }
    fclose(f);
    return 0;
}
