// Restriction-site counts of a FASTA file on the device (include/bin3c_b200.h: b3c_sites_*): per sequence its length,
// its site count (or head and tail site counts of a tip-based map) and its header bytes, equal to what
// seq_sites.fasta_site_table computes on the host.  The state machine and the matcher are in sites.cuh; this file
// launches them over one slab of file bytes at a time:
//   k_tiles    one thread per 32-byte chunk: the chunk's function of its entry class (sites.cuh: Fn), composed per
//              8 KB tile
//   k_prefix   one block: the exclusive scan of the tile functions, and the slab summary (kept bytes, headers,
//              name bytes, the pending whitespace run, room in the table and the name arena)
//   k_emit     one thread per chunk again: its entry state from the scans, then kept masks, name bytes and one table
//              row per header
//   k_match    one thread per kept position: all patterns at once on a window of 16 masks, warp-aggregated adds to
//              the sequence's int64 counter
//   k_close    tip maps, one warp per sequence that ends in the slab: head and tail windows
//   k_save     tip maps: the first and last tip_size masks of the sequence open at the slab end
//   k_commit   one thread: the state carried to the next slab
// Nothing is written when the table or the arena is too small (B3C_ERR_CAPACITY): the caller grows them and repeats
// the slab.
#include <algorithm>

#include "common.cuh"
#include "sites.cuh"

namespace b3c {
namespace {

using namespace b3c_sites;

constexpr unsigned long long NO_ERR = ~0ull;
constexpr int SCAN_THREADS = 512;
constexpr int MAX_GRID = kNumSMs * 8;

struct Header {
    Patterns P;
    State st;
    SlabInfo si;
    int64_t tip;
    unsigned long long err;          // (file offset << 8) | byte of the first byte >= 0x80 in a sequence line
};

struct Layout {
    int64_t slab, tip, n_tiles;
    int64_t fn_off, pre_off, k_off, head_off, ring_off, bytes;
};
std::mutex g_mu;
std::unordered_map<const void *, Layout> g_layouts;

Layout layout_for(int64_t slab, int64_t tip) {
    Layout L;
    Carver c;
    L.slab = slab;
    L.tip = tip;
    L.n_tiles = ceil_div(slab, TILE_BYTES);
    c.take(sizeof(Header));
    L.fn_off = c.take(L.n_tiles * (int64_t)sizeof(Fn));
    L.pre_off = c.take(L.n_tiles * (int64_t)sizeof(Fn));
    L.k_off = c.take(slab);
    L.head_off = c.take(tip > 0 ? tip : 1);
    L.ring_off = c.take(tip > 0 ? tip : 1);
    L.bytes = c.cur;
    return L;
}

// exclusive scan of one Fn per thread (Hillis-Steele in shared memory); *total gets the composition of all
template <int N>
__device__ Fn block_scan_fn(const Fn &v, Fn *sm, Fn *total) {
    const int t = threadIdx.x;
    sm[t] = v;
    __syncthreads();
    for (int off = 1; off < N; off <<= 1) {
        const Fn x = t >= off ? fn_compose(sm[t - off], sm[t]) : sm[t];
        __syncthreads();
        sm[t] = x;
        __syncthreads();
    }
    const Fn r = t > 0 ? sm[t - 1] : fn_identity();
    *total = sm[N - 1];
    __syncthreads();
    return r;
}

__device__ __forceinline__ Fn chunk_of(const uint8_t *buf, int64_t n, uint8_t prev, int64_t c) {
    const int64_t p0 = c * CHUNK;
    return p0 < n ? chunk_fn(buf, p0, p0 + CHUNK < n ? p0 + CHUNK : n, prev) : fn_identity();
}

__global__ void __launch_bounds__(TILE_THREADS) k_tiles(const uint8_t *buf, int64_t n, const Header *hd, Fn *tile_fn) {
    __shared__ Fn sm[TILE_THREADS];
    const Fn f = chunk_of(buf, n, hd->st.prev, (int64_t)blockIdx.x * TILE_THREADS + threadIdx.x);
    Fn total;
    block_scan_fn<TILE_THREADS>(f, sm, &total);
    if (threadIdx.x == 0) tile_fn[blockIdx.x] = total;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_prefix(Header *hd, const Fn *tile_fn, Fn *tile_pre, int64_t n_tiles,
                                                         int64_t n, int64_t seq_cap, int64_t name_cap) {
    __shared__ Fn sm[SCAN_THREADS];
    const int64_t per = (n_tiles + SCAN_THREADS - 1) / SCAN_THREADS;
    const int64_t lo = min((int64_t)threadIdx.x * per, n_tiles), hi = min(lo + per, n_tiles);
    Fn agg = fn_identity();
    for (int64_t i = lo; i < hi; ++i) agg = fn_compose(agg, tile_fn[i]);
    Fn total;
    Fn p = block_scan_fn<SCAN_THREADS>(agg, sm, &total);
    for (int64_t i = lo; i < hi; ++i) {
        tile_pre[i] = p;
        p = fn_compose(p, tile_fn[i]);
    }
    if (threadIdx.x == 0) hd->si = summarize(hd->st, total, n, hd->P.lmax, seq_cap, name_cap);
}

__global__ void __launch_bounds__(TILE_THREADS) k_emit(const uint8_t *buf, int64_t n, Header *hd, const Fn *tile_pre,
                                                       uint8_t *K, uint8_t *names, int64_t *rows) {
    __shared__ Fn sm[TILE_THREADS];
    if (hd->si.overflow) return;
    const uint8_t prev = hd->st.prev;
    const int64_t c = (int64_t)blockIdx.x * TILE_THREADS + threadIdx.x;
    Fn total;
    const Fn ex = block_scan_fn<TILE_THREADS>(chunk_of(buf, n, prev, c), sm, &total);
    const int64_t p0 = c * CHUNK;
    if (p0 >= n) return;
    Entry e0;
    e0.cls = hd->st.cls;
    e0.pend = e0.k = e0.a = e0.j = 0;
    const Entry e = fn_apply(fn_compose(tile_pre[blockIdx.x], ex), e0);
    const int64_t bad = emit_chunk(buf, p0, p0 + CHUNK < n ? p0 + CHUNK : n, prev, e, hd->si, K, names, rows);
    if (bad >= 0) atomicMin(&hd->err, ((unsigned long long)(hd->st.off + bad) << 8) | buf[bad]);
}

__global__ void __launch_bounds__(256) k_match(const Header *hd, const uint8_t *K, int64_t *rows) {
    __shared__ Patterns P;
    __shared__ SlabInfo s;
    if (threadIdx.x == 0) {
        P = hd->P;
        s = hd->si;
    }
    __syncthreads();
    if (s.overflow || P.n == 0) return;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x - (P.lmax - 1); base < s.m; base += stride) {
        int64_t c = 0;
        const int64_t row = count_at(P, s, K, rows, base + threadIdx.x, &c);
        const long long key = c > 0 ? row : -1;
        const unsigned peers = __match_any_sync(kFullMask, key);
        const unsigned sum = __reduce_add_sync(peers, (unsigned)c);
        if (key >= 0 && (int)lane_id() == __ffs(peers) - 1)
            atomicAdd((unsigned long long *)&rows[key * N_COLS + COL_CNT], (unsigned long long)sum);
    }
}

// one warp: head and tail sites of the sequence in table row `row`, n bytes long
__device__ void close_tips(const Patterns &P, const SeqView &v, int64_t n, int64_t *row) {
    int64_t w[4];
    tip_windows(n, v.tip, w);
    const unsigned lane = lane_id();
    long long hc = 0, tc = 0;
    for (int64_t q = w[0] + lane; q < w[1]; q += 32) hc += window_count_at(P, v, w[0], w[1], q);
    for (int64_t q = w[2] + lane; q < w[3]; q += 32) tc += window_count_at(P, v, w[2], w[3], q);
    hc = warp_sum(hc);
    tc = warp_sum(tc);
    if (lane == 0) {
        row[COL_HEAD] = hc;
        row[COL_TAIL] = tc;
    }
}

__global__ void __launch_bounds__(256) k_close(const Header *hd, const uint8_t *K, int64_t *rows, const uint8_t *head,
                                               const uint8_t *ring) {
    __shared__ Patterns P;
    __shared__ SlabInfo s;
    if (threadIdx.x == 0) {
        P = hd->P;
        s = hd->si;
    }
    __syncthreads();
    if (s.overflow) return;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < s.nnew; w += warps) {
        const int64_t r = s.nseq0 + w - 1;           // header w closes the sequence before it
        if (r < 0) continue;
        const int64_t g = rows[r * N_COLS + COL_G];
        close_tips(P, seq_view(s, K, g, head, ring, hd->tip), rows[(r + 1) * N_COLS + COL_G] - g, rows + r * N_COLS);
    }
}

__global__ void __launch_bounds__(256) k_save(const Header *hd, const uint8_t *K, const int64_t *rows, uint8_t *head,
                                              uint8_t *ring) {
    const SlabInfo &s = hd->si;
    if (s.overflow) return;
    const int64_t nseq = s.nseq0 + s.nnew;
    if (nseq == 0) return;
    const int64_t g = rows[(nseq - 1) * N_COLS + COL_G];
    const SeqView v = seq_view(s, K, g, head, ring, hd->tip);
    const int64_t L = s.Gbase + s.m - g;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < v.tip; t += (int64_t)gridDim.x * blockDim.x)
        save_slot(v, L, t, head, ring);
}

__global__ void k_commit(Header *hd, const uint8_t *buf, const uint8_t *K, const int64_t *rows) {
    if (hd->si.overflow) return;
    commit(hd->st, hd->si, buf, K, rows, hd->P.lmax);
}

// at the end of the file: the head and tail sites of the last sequence, from its saved bytes
__global__ void k_close_last(const Header *hd, int64_t *rows, const uint8_t *head, const uint8_t *ring) {
    const State &st = hd->st;
    SlabInfo s;
    s.n = 0;
    s.G0 = s.Gbase = st.G;
    s.m = 0;
    const int64_t r = st.nseq - 1;
    const int64_t g = rows[r * N_COLS + COL_G];
    close_tips(hd->P, seq_view(s, nullptr, g, head, ring, hd->tip), st.G - g, rows + r * N_COLS);
}

__global__ void k_rows(const Header *hd, const int64_t *rows, int64_t *out) {
    const State &st = hd->st;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < st.nseq; i += (int64_t)gridDim.x * blockDim.x)
        finish_row(rows, i, st.nseq, st.G, st.A, hd->tip > 0, out);
}

bool find_layout(const void *ws, Layout *L) {
    std::lock_guard<std::mutex> g(g_mu);
    auto it = g_layouts.find(ws);
    if (it == g_layouts.end()) return false;
    *L = it->second;
    return true;
}

}  // namespace
}  // namespace b3c

using namespace b3c;

extern "C" {

int64_t b3c_sites_workspace_bytes(int64_t slab_bytes, int32_t tip_size) {
    if (slab_bytes < 1 || slab_bytes > B3C_SITES_MAX_SLAB || tip_size < 0) {
        set_error("b3c_sites_workspace_bytes: slab_bytes must be in [1, %lld] and tip_size non-negative",
                  (long long)B3C_SITES_MAX_SLAB);
        return B3C_ERR_ARG;
    }
    return layout_for(slab_bytes, tip_size).bytes;
}

int b3c_sites_begin(void *d_ws, int64_t ws_bytes, int64_t slab_bytes, const uint8_t *h_masks, const int32_t *h_lengths,
                    const int32_t *h_weights, int32_t n_patterns, int32_t tip_size, void *stream) {
    B3C_REQUIRE(d_ws != nullptr, "b3c_sites_begin: null workspace");
    B3C_REQUIRE(slab_bytes >= 1 && slab_bytes <= B3C_SITES_MAX_SLAB && tip_size >= 0,
                "b3c_sites_begin: slab_bytes must be in [1, %lld] and tip_size non-negative", (long long)B3C_SITES_MAX_SLAB);
    B3C_REQUIRE(n_patterns >= 0 && n_patterns <= B3C_SITES_MAX_PATTERNS,
                "b3c_sites_begin: %d patterns, at most %d distinct ones are supported", n_patterns, B3C_SITES_MAX_PATTERNS);
    B3C_REQUIRE(n_patterns == 0 || (h_masks && h_lengths && h_weights), "b3c_sites_begin: null pattern table");
    const Layout L = layout_for(slab_bytes, tip_size);
    B3C_REQUIRE(ws_bytes >= L.bytes, "b3c_sites_begin: workspace holds %lld bytes, needs %lld", (long long)ws_bytes,
                (long long)L.bytes);
    Header h;
    memset(&h, 0, sizeof(h));
    h.P.n = n_patterns;
    h.P.lmax = 1;
    for (int p = 0; p < n_patterns; ++p) {
        const int len = h_lengths[p];
        B3C_REQUIRE(len >= 1 && len <= B3C_SITES_MAX_LEN, "b3c_sites_begin: pattern %d has %d bases, the counter takes "
                    "1 to %d", p, len, B3C_SITES_MAX_LEN);
        B3C_REQUIRE(h_weights[p] >= 1, "b3c_sites_begin: pattern %d has weight %d", p, h_weights[p]);
        uint64_t word = 0, full = 0;
        for (int i = 0; i < len; ++i) {
            const uint8_t m = h_masks[p * B3C_SITES_MAX_LEN + i];
            B3C_REQUIRE(m >= 1 && m <= 15, "b3c_sites_begin: pattern %d base %d has mask %d", p, i, m);
            word |= (uint64_t)m << (4 * i);
            full |= 1ull << (4 * i);
        }
        h.P.word[p] = word;
        h.P.full[p] = full;
        h.P.len[p] = len;
        h.P.weight[p] = h_weights[p];
        if (len > h.P.lmax) h.P.lmax = len;
    }
    h.st = state_initial();
    h.tip = tip_size;
    h.err = NO_ERR;
    cudaStream_t s = (cudaStream_t)stream;
    B3C_CUDA(cudaMemcpyAsync(d_ws, &h, sizeof(h), cudaMemcpyHostToDevice, s));
    B3C_CUDA(cudaStreamSynchronize(s));               // h lives on this stack
    std::lock_guard<std::mutex> g(g_mu);
    g_layouts[d_ws] = L;
    return B3C_OK;
}

int b3c_sites_slab(void *d_ws, const uint8_t *d_bytes, int64_t n_bytes, int64_t *d_seqs, int64_t seq_capacity,
                   uint8_t *d_names, int64_t names_capacity, int64_t *h_result, void *stream) {
    Layout L;
    B3C_REQUIRE(find_layout(d_ws, &L), "b3c_sites_slab: call b3c_sites_begin on this workspace first");
    B3C_REQUIRE(n_bytes >= 1 && n_bytes <= L.slab, "b3c_sites_slab: %lld bytes, the workspace takes 1 to %lld",
                (long long)n_bytes, (long long)L.slab);
    B3C_REQUIRE(d_bytes && h_result && seq_capacity >= 0 && names_capacity >= 0 && (seq_capacity == 0 || d_seqs) &&
                    (names_capacity == 0 || d_names),
                "b3c_sites_slab: null argument");
    cudaStream_t s = (cudaStream_t)stream;
    uint8_t *ws = (uint8_t *)d_ws;
    Header *hd = (Header *)ws;
    Fn *tile_fn = (Fn *)(ws + L.fn_off), *tile_pre = (Fn *)(ws + L.pre_off);
    uint8_t *K = ws + L.k_off, *head = ws + L.head_off, *ring = ws + L.ring_off;
    const int64_t n_tiles = ceil_div(n_bytes, TILE_BYTES);
    B3C_CUDA(cudaMemsetAsync(K, 0, (size_t)n_bytes, s));
    k_tiles<<<(unsigned)n_tiles, TILE_THREADS, 0, s>>>(d_bytes, n_bytes, hd, tile_fn);
    B3C_LAUNCH_CHECK();
    k_prefix<<<1, SCAN_THREADS, 0, s>>>(hd, tile_fn, tile_pre, n_tiles, n_bytes, seq_capacity, names_capacity);
    B3C_LAUNCH_CHECK();
    k_emit<<<(unsigned)n_tiles, TILE_THREADS, 0, s>>>(d_bytes, n_bytes, hd, tile_pre, K, d_names, d_seqs);
    B3C_LAUNCH_CHECK();
    k_match<<<(unsigned)std::min<int64_t>(ceil_div(n_bytes + MAX_LEN, 256), MAX_GRID), 256, 0, s>>>(hd, K, d_seqs);
    B3C_LAUNCH_CHECK();
    if (L.tip > 0) {
        k_close<<<(unsigned)std::min<int64_t>(ceil_div(n_bytes / 2 + 1, 8), MAX_GRID), 256, 0, s>>>(hd, K, d_seqs, head,
                                                                                                  ring);
        B3C_LAUNCH_CHECK();
        k_save<<<(unsigned)std::min<int64_t>(ceil_div(L.tip, 256), MAX_GRID), 256, 0, s>>>(hd, K, d_seqs, head, ring);
        B3C_LAUNCH_CHECK();
    }
    k_commit<<<1, 1, 0, s>>>(hd, d_bytes, K, d_seqs);
    B3C_LAUNCH_CHECK();
    struct {
        SlabInfo si;
        State st;
        unsigned long long err;
    } r;
    B3C_CUDA(cudaMemcpyAsync(&r.si, &hd->si, sizeof(r.si), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaMemcpyAsync(&r.st, &hd->st, sizeof(r.st), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaMemcpyAsync(&r.err, &hd->err, sizeof(r.err), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaStreamSynchronize(s));
    if (r.err != NO_ERR) {
        set_error("byte 0x%02x at file offset %llu lies in a sequence line: text-mode lengths count characters, "
                  "not bytes", (unsigned)(r.err & 0xff), r.err >> 8);
        return B3C_ERR_FORMAT;
    }
    if (r.si.overflow) {
        h_result[0] = r.si.nseq0 + r.si.nnew;
        h_result[1] = r.si.A0 + r.si.na;
        h_result[2] = r.st.G;
        set_error("b3c_sites_slab: the slab needs %lld table rows and %lld name bytes, there are %lld and %lld",
                  (long long)h_result[0], (long long)h_result[1], (long long)seq_capacity, (long long)names_capacity);
        return B3C_ERR_CAPACITY;
    }
    h_result[0] = r.st.nseq;
    h_result[1] = r.st.A;
    h_result[2] = r.st.G;
    return B3C_OK;
}

int b3c_sites_finish(void *d_ws, int64_t *d_seqs, int64_t *d_out, int64_t out_rows, int64_t *h_result, void *stream) {
    Layout L;
    B3C_REQUIRE(find_layout(d_ws, &L), "b3c_sites_finish: call b3c_sites_begin on this workspace first");
    B3C_REQUIRE(h_result != nullptr, "b3c_sites_finish: null argument");
    cudaStream_t s = (cudaStream_t)stream;
    uint8_t *ws = (uint8_t *)d_ws;
    const Header *hd = (const Header *)ws;
    State st;
    B3C_CUDA(cudaMemcpyAsync(&st, &hd->st, sizeof(st), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaStreamSynchronize(s));
    B3C_REQUIRE(out_rows >= st.nseq && (st.nseq == 0 || (d_seqs && d_out)),
                "b3c_sites_finish: %lld sequences, the output holds %lld", (long long)st.nseq, (long long)out_rows);
    if (st.nseq > 0) {
        if (L.tip > 0) {
            k_close_last<<<1, 32, 0, s>>>(hd, d_seqs, ws + L.head_off, ws + L.ring_off);
            B3C_LAUNCH_CHECK();
        }
        k_rows<<<(unsigned)std::min<int64_t>(ceil_div(st.nseq, 256), MAX_GRID), 256, 0, s>>>(hd, d_seqs, d_out);
        B3C_LAUNCH_CHECK();
        B3C_CUDA(cudaStreamSynchronize(s));
    }
    h_result[0] = st.nseq;
    h_result[1] = st.A;
    h_result[2] = st.G;
    return B3C_OK;
}

}  // extern "C"
