// Host build of the device edge-list formatter (bin3c_b200/csrc/edgefmt.cuh), for tests/test_edgefmt_cpu.py.  Each line
// is measured, then written into a buffer of the line bound, as the kernels of edgefmt.cu do it.
//   edgefmt_check <in file> <out file>
// in file: int64 n, int32 separator byte, int32 float style, int32 u[n], int32 v[n], float64 w[n].
// out file: the text.  A line whose written length differs from its measured length, or exceeds the bound, exits 3.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../bin3c_b200/csrc/edgefmt.cuh"

using namespace b3c_edgefmt;

int main(int argc, char **argv) {
    if (argc != 3) return 2;
    FILE *f = fopen(argv[1], "rb");
    if (!f) return 2;
    int64_t n = 0;
    int32_t sep = 0, style = 0;
    if (fread(&n, 8, 1, f) != 1 || fread(&sep, 4, 1, f) != 1 || fread(&style, 4, 1, f) != 1 || n < 0) return 2;
    std::vector<int32_t> u(n), v(n);
    std::vector<double> w(n);
    if (fread(u.data(), 4, n, f) != (size_t)n || fread(v.data(), 4, n, f) != (size_t)n ||
        fread(w.data(), 8, n, f) != (size_t)n)
        return 2;
    fclose(f);
    const Pow5 T{POW5_SPLIT, POW5_INV_SPLIT};
    std::vector<char> out;
    out.reserve((size_t)n * 32);
    char line[MAX_LINE_BYTES + 8];
    for (int64_t i = 0; i < n; ++i) {
        const Line L = line_measure(u[i], v[i], w[i], style, T);
        const int b = L.bytes();
        memset(line, 0x55, sizeof(line));
        line_put(L, u[i], v[i], (char)sep, style, line);
        if (b > MAX_LINE_BYTES || line[b - 1] != '\n' || line[b] != 0x55) {
            printf("ERR %lld %d\n", (long long)i, b);
            return 3;
        }
        out.insert(out.end(), line, line + b);
    }
    FILE *o = fopen(argv[2], "wb");
    if (!o || fwrite(out.data(), 1, out.size(), o) != out.size() || fclose(o) != 0) return 2;
    return 0;
}
