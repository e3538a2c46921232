// Host build of the device site counter's state machine and matcher (bin3c_b200/csrc/sites.cuh), for
// tests/test_sites_cpu.py.  It runs the steps of sites.cu one after the other, each kernel's threads as a loop, over
// slabs cut at the given sizes, and writes the table b3c_sites_finish returns.
//   sites_check <fasta bytes> <pattern file> <tip_size> <cut> <out file>
// pattern file: int32 n, then per pattern int32 length, int32 weight, 16 mask bytes.  cut: a slab size in bytes, or
// r<seed> for slabs of random sizes in [1, 64].  out file: int64 sequences, int64 name bytes, int64[sequences][5] as
// b3c_sites_finish, then the name arena.  A byte >= 0x80 in a sequence line prints "ERR <offset> <byte>", exits 3.
#include <cinttypes>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <random>
#include <vector>

#include "../../bin3c_b200/csrc/sites.cuh"

using namespace b3c_sites;

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

static void close_tips(const Patterns &P, const SeqView &v, int64_t n, int64_t *row) {
    int64_t w[4];
    tip_windows(n, v.tip, w);
    int64_t hc = 0, tc = 0;
    for (int64_t q = w[0]; q < w[1]; ++q) hc += window_count_at(P, v, w[0], w[1], q);
    for (int64_t q = w[2]; q < w[3]; ++q) tc += window_count_at(P, v, w[2], w[3], q);
    row[COL_HEAD] = hc;
    row[COL_TAIL] = tc;
}

int main(int argc, char **argv) {
    if (argc != 6) return 2;
    const std::vector<uint8_t> data = slurp(argv[1]);
    const std::vector<uint8_t> pf = slurp(argv[2]);
    const int64_t tip = atoll(argv[3]);
    Patterns P;
    memset(&P, 0, sizeof(P));
    int32_t np;
    memcpy(&np, pf.data(), 4);
    P.n = np;
    P.lmax = 1;
    for (int p = 0; p < np; ++p) {
        const uint8_t *e = pf.data() + 4 + p * 24;
        memcpy(&P.len[p], e, 4);
        memcpy(&P.weight[p], e + 4, 4);
        for (int i = 0; i < P.len[p]; ++i) {
            P.word[p] |= (uint64_t)e[8 + i] << (4 * i);
            P.full[p] |= 1ull << (4 * i);
        }
        if (P.len[p] > P.lmax) P.lmax = P.len[p];
    }
    const bool random_cuts = argv[4][0] == 'r';
    std::mt19937_64 rng(random_cuts ? atoll(argv[4] + 1) : 0);
    const int64_t cut = random_cuts ? 0 : atoll(argv[4]);

    const int64_t size = (int64_t)data.size();
    const int64_t seq_cap = size + 1, name_cap = size + 1;
    std::vector<int64_t> rows(N_COLS * (seq_cap + 1));
    std::vector<uint8_t> names(name_cap), head(tip > 0 ? tip : 1), ring(tip > 0 ? tip : 1);
    State st = state_initial();
    for (int64_t off = 0; off < size;) {
        int64_t n = random_cuts ? 1 + (int64_t)(rng() % 64) : cut;
        if (n > size - off) n = size - off;
        const uint8_t *buf = data.data() + off;
        // k_tiles
        const int64_t n_chunks = (n + CHUNK - 1) / CHUNK, n_tiles = (n + TILE_BYTES - 1) / TILE_BYTES;
        std::vector<Fn> cf(n_chunks), tf(n_tiles, fn_identity()), tp(n_tiles);
        for (int64_t c = 0; c < n_chunks; ++c) {
            cf[c] = chunk_fn(buf, c * CHUNK, std::min<int64_t>(n, (c + 1) * CHUNK), st.prev);
            tf[c / TILE_THREADS] = fn_compose(tf[c / TILE_THREADS], cf[c]);
        }
        // k_prefix
        Fn acc = fn_identity();
        for (int64_t t = 0; t < n_tiles; ++t) {
            tp[t] = acc;
            acc = fn_compose(acc, tf[t]);
        }
        const SlabInfo s = summarize(st, acc, n, P.lmax, seq_cap, name_cap);
        if (s.overflow) return 4;
        // k_emit
        std::vector<uint8_t> K(n, 0);
        Fn in = fn_identity();
        for (int64_t c = 0; c < n_chunks; ++c) {
            if (c % TILE_THREADS == 0) in = tp[c / TILE_THREADS];
            Entry e0;
            e0.cls = st.cls;
            e0.pend = e0.k = e0.a = e0.j = 0;
            const int64_t bad = emit_chunk(buf, c * CHUNK, std::min<int64_t>(n, (c + 1) * CHUNK), st.prev,
                                           fn_apply(in, e0), s, K.data(), names.data(), rows.data());
            if (bad >= 0) {
                printf("ERR %" PRId64 " %d\n", st.off + bad, buf[bad]);
                return 3;
            }
            in = fn_compose(in, cf[c]);
        }
        // k_match
        for (int64_t pos = -(int64_t)(P.lmax - 1); pos < s.m; ++pos) {
            int64_t c;
            const int64_t row = count_at(P, s, K.data(), rows.data(), pos, &c);
            if (row >= 0) rows[row * N_COLS + COL_CNT] += c;
        }
        if (tip > 0) {
            // k_close
            for (int64_t w = 0; w < s.nnew; ++w) {
                const int64_t r = s.nseq0 + w - 1;
                if (r < 0) continue;
                const int64_t g = rows[r * N_COLS + COL_G];
                close_tips(P, seq_view(s, K.data(), g, head.data(), ring.data(), tip),
                           rows[(r + 1) * N_COLS + COL_G] - g, &rows[r * N_COLS]);
            }
            // k_save
            const int64_t nseq = s.nseq0 + s.nnew;
            if (nseq > 0) {
                const int64_t g = rows[(nseq - 1) * N_COLS + COL_G];
                const SeqView v = seq_view(s, K.data(), g, head.data(), ring.data(), tip);
                for (int64_t t = 0; t < tip; ++t) save_slot(v, s.Gbase + s.m - g, t, head.data(), ring.data());
            }
        }
        commit(st, s, buf, K.data(), rows.data(), P.lmax);
        off += n;
    }
    // b3c_sites_finish
    if (st.nseq > 0 && tip > 0) {
        SlabInfo s;
        memset(&s, 0, sizeof(s));
        s.G0 = s.Gbase = st.G;
        const int64_t r = st.nseq - 1, g = rows[r * N_COLS + COL_G];
        close_tips(P, seq_view(s, nullptr, g, head.data(), ring.data(), tip), st.G - g, &rows[r * N_COLS]);
    }
    std::vector<int64_t> out(5 * (st.nseq > 0 ? st.nseq : 1));
    for (int64_t i = 0; i < st.nseq; ++i) finish_row(rows.data(), i, st.nseq, st.G, st.A, tip > 0, out.data());
    FILE *f = fopen(argv[5], "wb");
    if (!f) return 2;
    fwrite(&st.nseq, 8, 1, f);
    fwrite(&st.A, 8, 1, f);
    fwrite(out.data(), 8, 5 * st.nseq, f);
    fwrite(names.data(), 1, st.A, f);
    fclose(f);
    return 0;
}
