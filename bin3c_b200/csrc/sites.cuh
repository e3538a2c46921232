// Restriction-site counting of a FASTA byte stream, written once for the device counter (sites.cu) and for a plain
// C++ build on the host (tests/native/sites_check.cpp drives it serially over arbitrary slab cuts and
// tests/test_sites_cpu.py compares the result with seq_sites.fasta_site_table).
//
// The specification is the host counter: the file read in text mode (universal newlines), a line is a header iff its
// first byte is '>', a sequence line contributes line.strip() upper-cased, sequences are joined per header, and every
// pattern is searched with overlaps.  Here that becomes a per-byte state machine over three line classes:
//   HDR   inside a header line: the bytes after '>' go to the name arena
//   LEAD  a sequence line before its first non-whitespace byte: whitespace is dropped
//   BODY  a sequence line after its first non-whitespace byte: whitespace is PENDING -- kept when another content
//         byte follows on the same line (internal whitespace), dropped at the line end (trailing whitespace)
// Kept bytes form the KEPT STREAM, one 4-bit base mask per byte (A 1, C 2, G 4, T 8, anything else 0, so whitespace,
// N and IUPAC letters match no pattern position).  Sequence j is the range [g_j, g_{j+1}) of the kept stream, and its
// name the range [a_j, a_{j+1}) of the name arena; bytes before the first header belong to no sequence.
//
// Parallel form.  A slab is cut into CHUNK-byte chunks; a chunk's effect on the state is a function Fn of the class
// it is entered in (whether a line starts at a byte depends only on that byte and the one before it), and Fn
// composes associatively, so a scan of chunk functions gives every chunk its entry state.  The pending run is the one
// unbounded piece of state: Fn says, per entry class, whether the run the chunk is entered with is kept, dropped or
// still pending at its end, so a run of any length crosses chunks and slabs as a count.
#pragma once

#include <stdint.h>

#ifdef __CUDACC__
#define B3C_SHD __host__ __device__ __forceinline__
#else
#define B3C_SHD inline
#endif

namespace b3c_sites {

constexpr int MAX_LEN = 16;          // longest pattern: one 64-bit word of 4-bit masks
constexpr int MAX_PATTERNS = 64;     // distinct patterns (a hit set is one 64-bit word)
constexpr int CHUNK = 32;            // bytes one thread classifies serially
constexpr int TILE_THREADS = 256;    // chunks per tile (one thread block)
constexpr int64_t TILE_BYTES = (int64_t)CHUNK * TILE_THREADS;

enum : int { HDR = 0, LEAD = 1, BODY = 2 };
// columns of the per-sequence table
enum : int { COL_G = 0, COL_A = 1, COL_CNT = 2, COL_HEAD = 3, COL_TAIL = 4, N_COLS = 5 };

B3C_SHD bool is_eol(uint8_t b) { return b == '\n' || b == '\r'; }
// str.strip() whitespace below 0x80
B3C_SHD bool is_ws(uint8_t b) { return (b >= 0x09 && b <= 0x0d) || (b >= 0x1c && b <= 0x20); }
// a line starts at b: after '\n', or after a '\r' that does not begin "\r\n"
B3C_SHD bool line_start(uint8_t prev, uint8_t b) { return prev == '\n' || (prev == '\r' && b != '\n'); }
B3C_SHD uint8_t base_mask(uint8_t b) {
    switch (b | 0x20) {
        case 'a': return 1;
        case 'c': return 2;
        case 'g': return 4;
        case 't': return 8;
        default: return 0;
    }
}

// A chunk's effect, for each class c it may be entered in: dk kept bytes (whitespace pending at entry excluded), dp the
// pending run it leaves that began inside it, da name bytes; dj header lines that start in it (the same for every c).
// f holds, for class c, in bits 4c..4c+3: the class at the end (2 bits), bit 2 "the entry's pending run is kept",
// bit 3 "the entry's pending run is still pending at the end".
struct Fn {
    int32_t dk[3], dp[3], da[3];
    int32_t dj;
    uint32_t f;
};

B3C_SHD Fn fn_identity() {
    Fn r;
    for (int c = 0; c < 3; ++c) r.dk[c] = r.dp[c] = r.da[c] = 0;
    r.dj = 0;
    r.f = (uint32_t)(0x8 | ((0x8 | 1) << 4) | ((0x8 | 2) << 8));
    return r;
}
B3C_SHD int fn_cls(const Fn &x, int c) { return (int)((x.f >> (4 * c)) & 3u); }
B3C_SHD bool fn_keeps(const Fn &x, int c) { return (x.f >> (4 * c + 2)) & 1u; }
B3C_SHD bool fn_passes(const Fn &x, int c) { return (x.f >> (4 * c + 3)) & 1u; }

// x, then y
B3C_SHD Fn fn_compose(const Fn &x, const Fn &y) {
    Fn r;
    r.f = 0;
    for (int c = 0; c < 3; ++c) {
        const int c1 = fn_cls(x, c);
        r.dk[c] = x.dk[c] + y.dk[c1] + (fn_keeps(y, c1) ? x.dp[c] : 0);
        r.dp[c] = (fn_passes(y, c1) ? x.dp[c] : 0) + y.dp[c1];
        r.da[c] = x.da[c] + y.da[c1];
        const uint32_t keeps = fn_keeps(x, c) || (fn_passes(x, c) && fn_keeps(y, c1));
        const uint32_t passes = fn_passes(x, c) && fn_passes(y, c1);
        r.f |= ((uint32_t)fn_cls(y, c1) | (keeps << 2) | (passes << 3)) << (4 * c);
    }
    r.dj = x.dj + y.dj;
    return r;
}

// the function of bytes [p0, p1) of a slab; prev = the byte before the slab (a line starts at the slab's first byte
// when it is '\n', also at the start of the file)
B3C_SHD Fn chunk_fn(const uint8_t *buf, int64_t p0, int64_t p1, uint8_t prev0) {
    Fn r;
    r.f = 0;
    r.dj = 0;
    for (int c = 0; c < 3; ++c) {
        int cls = c;
        int32_t k = 0, pend = 0, a = 0, j = 0;
        bool live = true, kept = false;              // the entry's pending run: still pending / kept
        for (int64_t p = p0; p < p1; ++p) {
            const uint8_t b = buf[p], prev = p > 0 ? buf[p - 1] : prev0;
            if (line_start(prev, b)) {
                live = false;
                pend = 0;
                if (b == '>') {
                    cls = HDR;
                    ++j;
                    continue;
                }
                cls = LEAD;
            }
            if (is_eol(b)) {
                live = false;
                pend = 0;
                continue;
            }
            if (cls == HDR) {
                ++a;
                continue;
            }
            if (is_ws(b)) {
                if (cls == BODY) ++pend;
                continue;
            }
            if (cls == BODY) {
                k += pend;
                if (live) kept = true;
            }
            live = false;
            pend = 0;
            ++k;
            cls = BODY;
        }
        r.dk[c] = k;
        r.dp[c] = pend;
        r.da[c] = a;
        r.dj = j;
        r.f |= ((uint32_t)cls | ((uint32_t)kept << 2) | ((uint32_t)live << 3)) << (4 * c);
    }
    return r;
}

// where a chunk starts: its class, the pending run (of this slab) it is entered with, and the kept, name and header
// counts of the slab before it
struct Entry {
    int32_t cls;
    int64_t pend, k, a, j;
};

B3C_SHD Entry fn_apply(const Fn &x, const Entry &e) {
    Entry r;
    const int c = e.cls;
    r.cls = fn_cls(x, c);
    r.k = e.k + x.dk[c] + (fn_keeps(x, c) ? e.pend : 0);
    r.pend = (fn_passes(x, c) ? e.pend : 0) + x.dp[c];
    r.a = e.a + x.da[c];
    r.j = e.j + x.dj;
    return r;
}

struct Patterns {
    uint64_t word[MAX_PATTERNS];     // nibble i = IUPAC mask of base i
    uint64_t full[MAX_PATTERNS];     // 0x1 in each of the pattern's nibbles
    int32_t len[MAX_PATTERNS];
    int32_t weight[MAX_PATTERNS];    // how many times the pattern is listed
    int32_t n, lmax;
};

// carried from slab to slab
struct State {
    int64_t G;                       // kept bytes so far (the pending run excluded)
    int64_t A;                       // name bytes so far
    int64_t nseq;                    // headers so far
    int64_t pend;                    // the pending whitespace run at the end of the last slab
    int64_t off;                     // file bytes so far
    int32_t cls;
    uint8_t prev;                    // the last byte of the last slab
    uint8_t carry[MAX_LEN];          // carry[i]: mask of kept position G - (lmax - 1) + i, 0 before the open sequence
};

B3C_SHD State state_initial() {
    State s;
    s.G = s.A = s.nseq = s.pend = s.off = 0;
    s.cls = LEAD;
    s.prev = '\n';
    for (int i = 0; i < MAX_LEN; ++i) s.carry[i] = 0;
    return s;
}

// one slab, from the composed function of all its chunks
struct SlabInfo {
    int64_t n;                       // bytes
    int64_t G0, Gbase;               // kept bytes before the slab; global position of the slab's first kept byte
    int64_t m;                       // kept bytes of the slab
    int64_t nseq0, nnew;             // headers before the slab, headers in it
    int64_t A0, na;                  // name bytes before, in the slab
    int64_t pend_out;
    int32_t cls_out;
    int32_t overflow;                // the table or the arena is too small: nothing is written
    uint8_t carry[MAX_LEN];          // carry[i]: kept position Gbase - (lmax - 1) + i
};

B3C_SHD SlabInfo summarize(const State &st, const Fn &total, int64_t n, int32_t lmax, int64_t seq_cap, int64_t name_cap) {
    SlabInfo s;
    const int c = st.cls;
    const int64_t kept_in = fn_keeps(total, c) ? st.pend : 0;  // the run pending at the slab start is kept
    s.n = n;
    s.G0 = st.G;
    s.Gbase = st.G + kept_in;
    s.m = total.dk[c];
    s.nseq0 = st.nseq;
    s.nnew = total.dj;
    s.A0 = st.A;
    s.na = total.da[c];
    s.pend_out = (fn_passes(total, c) ? st.pend : 0) + total.dp[c];
    s.cls_out = fn_cls(total, c);
    s.overflow = (s.nseq0 + s.nnew > seq_cap || s.A0 + s.na > name_cap) ? 1 : 0;
    // the kept run shifts the carried window: its bytes are whitespace (mask 0) of the open sequence
    const int w = lmax - 1;
    for (int i = 0; i < MAX_LEN; ++i) {
        const int64_t src = (int64_t)i + kept_in;
        s.carry[i] = (i < w && src < w) ? st.carry[src] : 0;
    }
    return s;
}

// the kept-stream mask at local position li of the slab (negative: the carried window; past m: 0)
B3C_SHD uint8_t kept_at(const SlabInfo &s, const uint8_t *K, int32_t lmax, int64_t li) {
    if (li >= s.m) return 0;
    if (li >= 0) return K[li];
    const int64_t ci = li + (lmax - 1);
    return ci >= 0 ? s.carry[ci] : 0;
}

// serial pass over one chunk from its entry: kept masks to K (pre-zeroed, local positions), name bytes to the arena,
// one table row per header.  Returns the slab position of a byte >= 0x80 in a sequence line, or -1.
B3C_SHD int64_t emit_chunk(const uint8_t *buf, int64_t p0, int64_t p1, uint8_t prev0, Entry e, const SlabInfo &s,
                           uint8_t *K, uint8_t *names, int64_t *rows) {
    int cls = e.cls;
    int64_t k = e.k, pend = e.pend, a = e.a, j = e.j;
    for (int64_t p = p0; p < p1; ++p) {
        const uint8_t b = buf[p], prev = p > 0 ? buf[p - 1] : prev0;
        if (line_start(prev, b)) {
            pend = 0;
            if (b == '>') {
                cls = HDR;
                int64_t *r = rows + (s.nseq0 + j) * N_COLS;
                r[COL_G] = s.Gbase + k;
                r[COL_A] = s.A0 + a;
                r[COL_CNT] = r[COL_HEAD] = r[COL_TAIL] = 0;
                ++j;
                continue;
            }
            cls = LEAD;
        }
        if (is_eol(b)) {
            pend = 0;
            continue;
        }
        if (cls == HDR) {
            names[s.A0 + a] = b;
            ++a;
            continue;
        }
        if (b >= 0x80) return p;
        if (is_ws(b)) {
            if (cls == BODY) ++pend;
            continue;
        }
        if (cls == BODY) k += pend;                  // internal whitespace: zeros already in K
        pend = 0;
        K[k++] = base_mask(b);
        cls = BODY;
    }
    return -1;
}

// nibbles of the window starting at local position s
B3C_SHD uint64_t window_at(const SlabInfo &s, const uint8_t *K, int32_t lmax, int64_t pos) {
    uint64_t w = 0;
    for (int i = 0; i < lmax; ++i) w |= (uint64_t)kept_at(s, K, lmax, pos + i) << (4 * i);
    return w;
}

// every one of the pattern's positions shares a bit with the window's mask
B3C_SHD bool matches(uint64_t win, uint64_t word, uint64_t full) {
    uint64_t x = win & word;
    x |= x >> 1;
    x |= x >> 2;
    return (x & full) == full;
}

B3C_SHD uint64_t hits(const Patterns &P, uint64_t win) {
    uint64_t h = 0;
    for (int p = 0; p < P.n; ++p)
        if (matches(win, P.word[p], P.full[p])) h |= 1ull << p;
    return h;
}

// the slab's header (local index 0 .. nnew-1) a kept byte at local position li belongs to; -1: the sequence open at
// the slab start
B3C_SHD int64_t header_of(const SlabInfo &s, const int64_t *rows, int64_t li) {
    const int64_t x = s.Gbase + li;
    int64_t lo = 0, hi = s.nnew;                      // count of headers with g <= x
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (rows[(s.nseq0 + mid) * N_COLS + COL_G] <= x) lo = mid + 1;
        else hi = mid;
    }
    return lo - 1;
}

// matches starting at local position pos whose last byte is in this slab, inside one sequence: adds to *count and
// returns the table row of that sequence (-1: none, or bytes before the first header)
B3C_SHD int64_t count_at(const Patterns &P, const SlabInfo &s, const uint8_t *K, const int64_t *rows, int64_t pos,
                         int64_t *count) {
    *count = 0;
    if (P.n == 0 || pos >= s.m || pos < -(int64_t)(P.lmax - 1)) return -1;
    const uint64_t h = hits(P, window_at(s, K, P.lmax, pos));
    if (!h) return -1;
    const int64_t hj = pos < 0 ? -1 : header_of(s, rows, pos);
    const int64_t row = s.nseq0 + hj;
    if (row < 0) return -1;
    const int64_t next = hj + 1 < s.nnew ? rows[(s.nseq0 + hj + 1) * N_COLS + COL_G] - s.Gbase : s.m;
    int64_t c = 0;
    for (int p = 0; p < P.n; ++p) {
        const int64_t end = pos + P.len[p] - 1;
        if (((h >> p) & 1) && end >= 0 && end < next) c += P.weight[p];
    }
    *count = c;
    return row;
}

// ---- tip windows -------------------------------------------------------------------------------------------------
// seq[:n//2] and seq[(-n)//2:] when n < 2 tip, else seq[:tip] and seq[-tip:]
B3C_SHD void tip_windows(int64_t n, int64_t tip, int64_t w[4]) {
    if (n < 2 * tip) {
        w[0] = 0, w[1] = n / 2, w[2] = n / 2, w[3] = n;
    } else {
        w[0] = 0, w[1] = tip, w[2] = n - tip, w[3] = n;
    }
}

// One sequence's bytes by sequence position q: this slab's kept bytes, the kept whitespace run the slab started with,
// then what was saved of earlier slabs: head[q] for q < tip, ring[q % tip] for the last tip positions.
struct SeqView {
    const uint8_t *K;
    int64_t m;
    int64_t loc0;                    // sequence position of local kept position 0
    int64_t qb;                      // positions below qb lie in earlier slabs
    const uint8_t *head, *ring;
    int64_t tip;
};

B3C_SHD SeqView seq_view(const SlabInfo &s, const uint8_t *K, int64_t g, const uint8_t *head, const uint8_t *ring,
                         int64_t tip) {
    SeqView v;
    v.K = K;
    v.m = s.m;
    v.loc0 = s.Gbase - g;
    v.qb = s.G0 > g ? s.G0 - g : 0;
    v.head = head;
    v.ring = ring;
    v.tip = tip;
    return v;
}

B3C_SHD uint8_t seq_at(const SeqView &v, int64_t q) {
    const int64_t li = q - v.loc0;
    if (li >= 0) return li < v.m ? v.K[li] : 0;
    if (q >= v.qb) return 0;
    return q < v.tip ? v.head[q] : v.ring[q % v.tip];
}

// matches starting at sequence position q that lie inside [lo, hi)
B3C_SHD int64_t window_count_at(const Patterns &P, const SeqView &v, int64_t lo, int64_t hi, int64_t q) {
    if (q < lo || q >= hi) return 0;
    uint64_t w = 0;
    for (int i = 0; i < P.lmax && q + i < hi; ++i) w |= (uint64_t)seq_at(v, q + i) << (4 * i);
    int64_t c = 0;
    for (int p = 0; p < P.n; ++p)
        if (q + P.len[p] <= hi && matches(w, P.word[p], P.full[p])) c += P.weight[p];
    return c;
}

// after the slab, slot t of the saved head and ring of the sequence open at its end (length L so far)
B3C_SHD void save_slot(const SeqView &v, int64_t L, int64_t t, uint8_t *head, uint8_t *ring) {
    if (t < v.tip && t >= v.qb && t < L) head[t] = seq_at(v, t);
    if (L > 0) {
        const int64_t q = L - 1 - ((L - 1 - t) % v.tip + v.tip) % v.tip;    // last position < L with q % tip == t
        if (q >= 0 && q >= v.qb) ring[t] = seq_at(v, q);
    }
}

// the state after the slab
B3C_SHD void commit(State &st, const SlabInfo &s, const uint8_t *buf, const uint8_t *K, const int64_t *rows,
                    int32_t lmax) {
    const int64_t G = s.Gbase + s.m, nseq = s.nseq0 + s.nnew;
    const int64_t g_open = nseq > 0 ? rows[(nseq - 1) * N_COLS + COL_G] : G;
    uint8_t c[MAX_LEN];
    for (int i = 0; i < MAX_LEN; ++i) {
        const int64_t pos = G - (lmax - 1) + i;
        c[i] = (i < lmax - 1 && pos >= g_open) ? kept_at(s, K, lmax, pos - s.Gbase) : 0;
    }
    for (int i = 0; i < MAX_LEN; ++i) st.carry[i] = c[i];
    st.G = G;
    st.A = s.A0 + s.na;
    st.nseq = nseq;
    st.pend = s.pend_out;
    st.cls = s.cls_out;
    if (s.n > 0) st.prev = buf[s.n - 1];
    st.off += s.n;
}

// the finished table: length, name range, sites (or head sites), tail sites
B3C_SHD void finish_row(const int64_t *rows, int64_t i, int64_t nseq, int64_t G, int64_t A, bool tips, int64_t *out) {
    const int64_t *r = rows + i * N_COLS;
    const int64_t g1 = i + 1 < nseq ? rows[(i + 1) * N_COLS + COL_G] : G;
    const int64_t a1 = i + 1 < nseq ? rows[(i + 1) * N_COLS + COL_A] : A;
    out[i * 5 + 0] = g1 - r[COL_G];
    out[i * 5 + 1] = r[COL_A];
    out[i * 5 + 2] = a1;
    out[i * 5 + 3] = tips ? r[COL_HEAD] : r[COL_CNT];
    out[i * 5 + 4] = tips ? r[COL_TAIL] : 0;
}

}  // namespace b3c_sites
