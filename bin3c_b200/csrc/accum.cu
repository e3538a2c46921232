// Pair accumulation: packed pair records -> exact-count canonical CSR (upper or symmetric).
//
// Replaces the per-pair Python loop of ContactMap._bin_map (contact_map.py:720-798), the
// tid->index dict (contact_map.py:818-832) and Sparse2DAccumulator.get_coo
// (sparse_utils.py:246-266).  Stages (all HBM-bound integer work, no tensor cores):
//
//   k_classify     one streaming pass over the records (8 B/pair).  tid -> index through a
//                  bitmap+rank table staged in shared memory (the reference assigns indices in
//                  BAM order, contact_map.py:545-564, so index = rank of tid among the kept
//                  references); exclusion test, then matcher bit (Q12); diagonal pairs are
//                  counted in a shared-memory histogram (most Hi-C pairs are intra-contig),
//                  off-diagonal pairs become keys (i << b | j), staged in shared memory and
//                  appended to the key buffer with one global atomic per 4096-record tile.
//   k_rs_*         LSD radix sort of the keys, 8-bit digits, only the 2b significant bits.
//   k_rle_*        run-length reduce of the sorted keys -> unique (i,j) + exact counts.
//   k_emit_*       upper and lower halves + diagonal scattered into canonical CSR; the lower
//                  half's order comes from a stable sort of (j, e) on j's bits alone.
#include <type_traits>

#include "common.cuh"

namespace b3c {

// ---- counters kept in the workspace ---------------------------------------------------
enum { C_NKEYS = 0, C_ACCEPT, C_EXCL, C_POOR, C_NNZ_UO, C_NNZ_DIAG, C_WEIGHT, C_LUT_OK, C_OVERFLOW, C_COUNT = 16 };

constexpr int CLS_THREADS = 1024;
constexpr int CLS_RPT = 4;                       // records per thread per tile (two 128-bit loads)
constexpr int CLS_WARPS = CLS_THREADS / 32;
constexpr int CLS_WTILE = 32 * CLS_RPT;          // 128 records = 1 KB of input per warp tile
constexpr int CLS_CAPW_MAX = 512;                // keys a warp stages before it flushes (at most)
constexpr int SMEM_MAX = 232448;                 // 227 KB opt-in limit per CTA on sm_100

constexpr int RS_THREADS = 512;
constexpr int RS_KPT = 8;
constexpr int RS_TILE = RS_THREADS * RS_KPT;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_BITS = 9;                       // widest digit (k_rs_*<9>); k_rs_*<8> where it needs no more passes
constexpr int RS_BINS = 1 << RS_BITS;            // sizes the histogram buffers
constexpr int RS_BLOCKS = kNumSMs * 4;

struct AccumState {
    int64_t cap = 0;
    int32_t n_seq = 0, n_refs = 0;
    int b = 0;                // bits per index in the key
    int64_t rank_words = 0;   // 64-bit words of the tid bitmap
    bool smem_diag = false;
    int smem_rank = 0;        // 0 gather, 1 pair table, 2 packed table, 3 two-level table (classify_tiles)
    int cls_smem = 0, cls_grid = 0, cls_cap_w = 0, cls_diag_k = 0;
    const int32_t *d_lut = nullptr;
    int64_t o_ctr, o_diag, o_bits, o_pref, o_keys_a, o_keys_b, o_uniq, o_pos, o_cnt, o_hist, o_heads,
        o_up_ptr, o_lo_ptr, o_len, o_indptr_f, o_indptr_u, o_scan_tmp, o_tmp64, total;
    bool reduced = false;
    int64_t nnz_uo = 0, nnz_diag = 0;
    int comp_in_a = 0;        // which key buffer holds the (j,i)-sorted composite after reduce
};

static std::mutex g_mu;
static std::unordered_map<void *, AccumState> g_states;

static int key_bits_for(int32_t n_seq) {
    int b = 1;
    while ((1ll << b) < (int64_t)n_seq) ++b;
    return b;
}

static void layout(AccumState &st) {
    Carver c;
    const int64_t cap = st.cap > 0 ? st.cap : 1;
    const int64_t n1 = (int64_t)st.n_seq + 1;
    st.o_ctr = c.take(C_COUNT * 8);
    st.o_diag = c.take((int64_t)st.n_seq * 4);
    st.o_bits = c.take(st.rank_words * 8);
    st.o_pref = c.take(st.rank_words * 4);
    st.o_tmp64 = c.take((st.rank_words + 1) * 8 * 2);
    st.o_keys_a = c.take(cap * 8);
    st.o_keys_b = c.take(cap * 8);
    st.o_uniq = c.take(cap * 8);
    st.o_pos = c.take((cap + 1) * 4);
    st.o_cnt = c.take(cap * 4);
    st.o_hist = c.take(((int64_t)RS_BINS * RS_BLOCKS + RS_BINS) * 4);
    st.o_heads = c.take((RS_BLOCKS + 2) * 8 * 2);
    st.o_up_ptr = c.take(n1 * 8);
    st.o_lo_ptr = c.take(n1 * 8);
    st.o_len = c.take(n1 * 8);
    st.o_indptr_f = c.take(n1 * 8);
    st.o_indptr_u = c.take(n1 * 8);
    int64_t m = st.n_seq > st.rank_words ? st.n_seq : st.rank_words;
    if (m < RS_BLOCKS) m = RS_BLOCKS;
    st.o_scan_tmp = c.take(scan_tmp_elems(m) * 8);
    st.total = c.cur;
}

static void plan(AccumState &st, int64_t cap, int32_t n_seq, int32_t n_refs) {
    st.cap = cap;
    st.n_seq = n_seq;
    st.n_refs = n_refs;
    st.b = key_bits_for(n_seq);
    st.rank_words = ceil_div(n_refs > 0 ? n_refs : 1, 64);
    // shared-memory plan of k_classify: per-warp key staging | rank table | diagonal histogram
    // (in shared memory the table is held as (32-bit word, prefix) pairs plus one zero sentinel)
    const int64_t rank64_bytes = align_up((st.rank_words * 2 + 1) * 8, 16);
    const int64_t rank32_bytes = align_up((ceil_div(n_refs > 0 ? n_refs : 1, 12) + 1) * 4, 16);
    // mode 3, for tables too long for the other two (C4: 1.1M references): the 64-bit bitmap words, a 16-bit prefix
    // per word relative to its block of 32 words, a 32-bit prefix per block -- 10.1 bytes per 64 references
    const int64_t rank3_bytes = align_up((st.rank_words + 1) * 8, 16) + align_up((st.rank_words + 1) * 2, 16) +
                                align_up((st.rank_words / 32 + 2) * 4, 16);
    const int64_t diag_bytes = align_up((int64_t)n_seq * 4, 16);
    // staging keys per warp that fit beside `fixed` bytes: at least one warp tile, at most CLS_CAPW_MAX
    auto cap_w = [](int64_t fixed, int key_bytes) -> int {
        int64_t c = (SMEM_MAX - fixed) / ((int64_t)CLS_WARPS * key_bytes);
        if (c > CLS_CAPW_MAX) c = CLS_CAPW_MAX;
        c &= ~(int64_t)31;
        return c >= CLS_WTILE ? (int)c : 0;
    };
    // the packed table (mode 2) where it fits with room for 256 staged keys per warp and the index fits its 20-bit
    // prefix; else the pair table (mode 1); else look-ups gather from global memory (mode 0)
    auto rank_mode = [&](int64_t other, int key_bytes, int64_t *bytes) -> int {
        if (st.b <= 20 && cap_w(other + rank32_bytes, key_bytes) >= 256) {
            *bytes = rank32_bytes;
            return 2;
        }
        if (cap_w(other + rank64_bytes, key_bytes)) {
            *bytes = rank64_bytes;
            return 1;
        }
        if (st.b <= 20 && cap_w(other + rank32_bytes, key_bytes)) {
            *bytes = rank32_bytes;
            return 2;
        }
        if (cap_w(other + rank3_bytes, key_bytes)) {
            *bytes = rank3_bytes;
            return 3;
        }
        *bytes = 0;
        return 0;
    };
    st.smem_diag = false;
    st.smem_rank = 0;
    int64_t fixed = 0, rb = 0;
    int kb = 8;
    if (st.b <= 16 && rank_mode(diag_bytes, 4, &rb)) {
        st.smem_diag = true;
        st.smem_rank = rank_mode(diag_bytes, 4, &rb);
        fixed = rb + diag_bytes;
        kb = 4;
    } else if (st.b <= 16 && cap_w(diag_bytes, 4)) {
        st.smem_diag = true;
        fixed = diag_bytes;
        kb = 4;
    } else {
        st.smem_rank = rank_mode(0, 8, &rb);
        fixed = rb;
    }
    st.cls_cap_w = cap_w(fixed, kb);
    st.cls_diag_k = 0;
    if (!st.smem_diag) {
        // a partial diagonal histogram in what is left beside the smallest staging, if it covers >= 5 % of the contigs
        const int64_t room = (SMEM_MAX - fixed - (int64_t)CLS_WARPS * CLS_WTILE * kb) / 4;
        if (room >= (int64_t)n_seq / 20 && room > 0) {
            st.cls_cap_w = CLS_WTILE;
            st.cls_diag_k = (int)(room < n_seq ? room : n_seq);
        }
    }
    st.cls_smem = (int)((int64_t)CLS_WARPS * st.cls_cap_w * kb + fixed + (int64_t)st.cls_diag_k * 4);
    st.cls_grid = kNumSMs;      // persistent: one 1024-thread CTA per SM, tiles strided over the grid
    layout(st);
}

// ---- rank table (bitmap + prefix popcount) -------------------------------------------------
__global__ void k_rank_bits(const int32_t *__restrict__ lut, int32_t n_refs, int64_t n_words,
                            unsigned long long *__restrict__ bits, int64_t *__restrict__ cnt) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_words) return;
    unsigned long long m = 0;
    const int64_t t0 = w * 64;
    for (int k = 0; k < 64; ++k) {
        const int64_t t = t0 + k;
        if (t < n_refs && lut[t] >= 0) m |= 1ull << k;
    }
    bits[w] = m;
    cnt[w] = __popcll(m);
}

__global__ void k_rank_verify(const int32_t *__restrict__ lut, int32_t n_refs, int32_t n_seq,
                              const unsigned long long *__restrict__ bits, const int64_t *__restrict__ pref64,
                              uint32_t *__restrict__ pref, int64_t n_words, unsigned long long *__restrict__ ctr) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n_words) pref[t] = (uint32_t)pref64[t];
    if (t >= n_refs) return;
    const int32_t v = lut[t];
    if (v < 0) return;
    const int64_t w = t >> 6;
    const int bit = (int)(t & 63);
    const int64_t expect = pref64[w] + __popcll(bits[w] & ((1ull << bit) - 1ull));
    if (expect != (int64_t)v || v >= n_seq) ctr[C_LUT_OK] = 0;   // benign race: every writer stores 0
}

// ---- classify ------------------------------------------------------------------------------
struct ClsParams {
    const uint64_t *rec;
    int64_t n_rec;
    int32_t rec_bytes;       // 8: native records; 5 or 6: narrow records (b3c_accum_add_pairs_packed)
    int32_t rec_same;        // 1: 3- or 4-byte records of pairs whose mates lie on ONE reference (b3c_accum_add_pairs_same)
    const int32_t *lut;
    int32_t n_refs, n_seq;
    int b;
    int64_t rank_words;
    const unsigned long long *g_bits;
    const uint32_t *g_pref;
    uint32_t *diag;
    uint64_t *keys;
    int64_t cap;
    unsigned long long *ctr;
    int cap_w;               // staging keys per warp
    int diag_k;              // without SMEM_DIAG: the first diag_k contigs' diagonal counters are in shared memory
};

// Every warp runs on its own: its own stream of 128-record warp tiles (strided over all warps of the grid, loads
// issued two tiles ahead), its own staging area of `cap_w` keys in shared memory and its own flushes -- one global
// atomic per flush reserves the run in the key buffer (the order of the keys does not matter: they are sorted next).
// There is no block barrier inside the loop.  The record logic is written without branches (look-ups read a zero
// sentinel word for out-of-table ids; exclusion, matcher and diagonal tests are predicates), because the four
// outcomes -- excluded, poor match, diagonal, off-diagonal -- are mixed in every warp and a branchy form executes
// all of them one after the other (it was 147 issued instructions per 32 records; this form is ~60).
// RANK: 0 = look-ups gather from the global tid -> index table; 1 = rank table in shared memory as (32-bit bitmap
// word, prefix) pairs, one 8-byte load per look-up; 2 = packed form, one 32-bit word per 12 references (12-bit bitmap,
// 20-bit prefix): a scattered 4-byte shared-memory load costs about half the wavefronts of an 8-byte one, and at C3
// the kernel is bound by the L1/shared-memory pipe (scattered diagonal REDs + table look-ups), not by issue or HBM.
template <bool SMEM_DIAG, int RANK>
__device__ __forceinline__ void classify_tiles(const ClsParams &P, unsigned char *smem) {
    using stage_t = typename std::conditional<SMEM_DIAG, uint32_t, uint64_t>::type;
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
    const unsigned lt = lanemask_lt();
    stage_t *s_stage = reinterpret_cast<stage_t *>(smem) + (size_t)warp * P.cap_w;
    unsigned char *cur = smem + sizeof(stage_t) * (size_t)CLS_WARPS * P.cap_w;
    const uint2 *s_tab = nullptr;
    const uint32_t *s_tab32 = nullptr;
    const uint32_t nw32 = (uint32_t)(P.rank_words * 2);
    const uint32_t nw12 = (uint32_t)((P.n_refs + 11) / 12);
    if (RANK == 1) {
        // the global table has 64-bit words with one prefix each; here it is re-cut into (32-bit word, prefix) pairs so
        // a look-up is ONE 8-byte shared-memory load, 32-bit shifts and a POPC; entry nw32 is the all-zero sentinel
        uint2 *tab = reinterpret_cast<uint2 *>(cur);
        cur += (((size_t)nw32 + 1) * 8 + 15) / 16 * 16;
        for (int64_t i = threadIdx.x; i < P.rank_words; i += CLS_THREADS) {
            const unsigned long long m = P.g_bits[i];
            const uint32_t lo = (uint32_t)m, hi = (uint32_t)(m >> 32), pf = P.g_pref[i];
            tab[2 * i] = make_uint2(lo, pf);
            tab[2 * i + 1] = make_uint2(hi, pf + __popc(lo));
        }
        if (threadIdx.x == 0) tab[nw32] = make_uint2(0u, 0u);
        s_tab = tab;
    }
    if (RANK == 2) {
        // word w covers references [12 w, 12 w + 12): bitmap in bits 0..11, rank of reference 12 w in bits 12..31
        uint32_t *tab = reinterpret_cast<uint32_t *>(cur);
        cur += (((size_t)nw12 + 1) * 4 + 15) / 16 * 16;
        for (uint32_t w = threadIdx.x; w < nw12; w += CLS_THREADS) {
            const uint32_t t0 = w * 12u;
            const int64_t q = t0 >> 6;
            const unsigned sh = t0 & 63u;
            const unsigned long long m0 = P.g_bits[q];
            unsigned long long m = m0 >> sh;
            if (sh > 52 && q + 1 < P.rank_words) m |= P.g_bits[q + 1] << (64 - sh);
            const uint32_t pf = P.g_pref[q] + (uint32_t)__popcll(m0 & ((1ull << sh) - 1ull));
            tab[w] = ((uint32_t)m & 0xfffu) | (pf << 12);
        }
        if (threadIdx.x == 0) tab[nw12] = 0u;
        s_tab32 = tab;
    }
    const unsigned long long *s_bits3 = nullptr;
    const uint16_t *s_rel3 = nullptr;
    const uint32_t *s_sup3 = nullptr;
    const uint32_t nw64 = (uint32_t)P.rank_words;
    if (RANK == 3) {
        // two-level form: word w (64 references) | its rank relative to block w / 32 (16 bit: < 2048) | the block's rank;
        // three shared-memory loads per look-up instead of a gather from global memory; entry nw64 is the zero sentinel
        unsigned long long *bits = reinterpret_cast<unsigned long long *>(cur);
        cur += (((size_t)nw64 + 1) * 8 + 15) / 16 * 16;
        uint16_t *rel = reinterpret_cast<uint16_t *>(cur);
        cur += (((size_t)nw64 + 1) * 2 + 15) / 16 * 16;
        uint32_t *sup = reinterpret_cast<uint32_t *>(cur);
        cur += (((size_t)nw64 / 32 + 2) * 4 + 15) / 16 * 16;
        for (uint32_t i = threadIdx.x; i < nw64; i += CLS_THREADS) {
            const uint32_t base = P.g_pref[i & ~31u];
            bits[i] = P.g_bits[i];
            rel[i] = (uint16_t)(P.g_pref[i] - base);
            if ((i & 31u) == 0) sup[i >> 5] = base;
        }
        if (threadIdx.x == 0) {
            bits[nw64] = 0ull;
            rel[nw64] = 0;
            if ((nw64 & 31u) == 0) sup[nw64 >> 5] = 0u;            // the sentinel opens a block of its own
        }
        s_bits3 = bits;
        s_rel3 = rel;
        s_sup3 = sup;
    }
    // diagonal counters of the first `dk` contigs live in shared memory (all of them with SMEM_DIAG; else as many as
    // fit beside the table and the staging: every one of them is a global RED less, and at C3 the kernel runs at
    // the rate the L2 retires the diagonal REDs -- 333M of them, ~140 G/s)
    uint32_t *s_diag = reinterpret_cast<uint32_t *>(cur);
    const uint32_t dk = SMEM_DIAG ? (uint32_t)P.n_seq : (uint32_t)P.diag_k;
    for (uint32_t i = threadIdx.x; i < dk; i += CLS_THREADS) s_diag[i] = 0;
    __syncthreads();

    unsigned n_ok = 0, n_valid = 0, n_acc = 0;
    unsigned cnt = 0;                                  // keys staged by this warp (warp-uniform)
    const int64_t n_tiles = (P.n_rec + CLS_WTILE - 1) / CLS_WTILE;
    const int64_t n_warps = (int64_t)gridDim.x * CLS_WARPS;
    const int64_t w0 = (int64_t)blockIdx.x * CLS_WARPS + warp;

    // index of a kept reference, or hit = false (excluded, or beyond the table); `on` = false skips the load
    auto lookup = [&](uint32_t t, bool on, bool &hit) -> uint32_t {
        if (RANK == 2) {
            uint32_t w = __umulhi(t, 0xAAAAAAABu) >> 3;             // t / 12
            const unsigned bit = t - w * 12u;
            w = min(w, nw12);
            uint32_t e = 0;
            if (on) e = s_tab32[w];
            hit = (e >> bit) & 1u;
            return (e >> 12) + __popc(e & ~(0xffffffffu << bit) & 0xfffu);
        } else if (RANK == 3) {
            const uint32_t w = min(t >> 6, nw64);
            unsigned long long m = 0ull;
            uint32_t pf = 0;
            if (on) {
                m = s_bits3[w];
                pf = (uint32_t)s_rel3[w] + s_sup3[w >> 5];
            }
            const unsigned bit = t & 63u;
            hit = (m >> bit) & 1ull;
            return pf + __popcll(m & ~(~0ull << bit));
        } else if (RANK == 1) {
            uint2 e = make_uint2(0u, 0u);
            if (on) e = s_tab[min(t >> 5, nw32)];
            const unsigned bit = t & 31u;
            hit = (e.x >> bit) & 1u;
            return e.y + __popc(e.x & ~(0xffffffffu << bit));
        } else {
            int32_t v = -1;
            if (on && t < (uint32_t)P.n_refs) v = __ldg(P.lut + t);
            hit = v >= 0 && v < P.n_seq;
            return (uint32_t)v;
        }
    };

    auto flush = [&]() {
        __syncwarp();
        unsigned long long gb = 0;
        if (lane == 0) gb = atomicAdd(&P.ctr[C_NKEYS], (unsigned long long)cnt);
        gb = __shfl_sync(kFullMask, gb, 0);
        if ((int64_t)(gb + cnt) <= P.cap) {
            for (unsigned i = lane; i < cnt; i += 32) P.keys[gb + i] = (uint64_t)s_stage[i];
        } else if (lane == 0) {
            P.ctr[C_OVERFLOW] = 1;
        }
        __syncwarp();
        cnt = 0;
    };

    // lane l of the warp reads records [base + h*64 + 2*l, +2) for h = 0, 1: two 128-bit streaming loads per tile
    auto load_tile = [&](int64_t tile, uint4 (&v)[CLS_RPT / 2]) -> unsigned {
        const int64_t base = tile * CLS_WTILE;
        if (P.rec_bytes == 8 && base + CLS_WTILE <= P.n_rec) {
#pragma unroll
            for (int h = 0; h < CLS_RPT / 2; ++h) v[h] = ld_stream_u4(P.rec + base + h * 64 + lane * 2);
            return (1u << CLS_RPT) - 1u;
        }
        unsigned okm = 0;
        if (P.rec_bytes != 8) {
            // narrow records: B bytes each, little endian, tid1 in bits [0, tb), the pass flag in bit tb, tid2 in
            // bits [tb + 1, 2 tb + 1), tb = (8 B - 1) / 2.  A record is cut out of the one or two 8-byte words that
            // hold it and widened to the native (lo, hi) halves, so the rest of the kernel does not change.
            // (same-reference records: one id in bits [0, 8 B - 1), the flag in the top bit; widened to tid1 = tid2)
            const int B = P.rec_bytes, tb = P.rec_same ? 8 * B - 1 : (8 * B - 1) / 2;
            const uint64_t tmask = (1ull << tb) - 1ull;
            const int64_t last_word = (P.n_rec * B - 1) >> 3;
#pragma unroll
            for (int h = 0; h < CLS_RPT / 2; ++h) {
                uint32_t q4[4] = {0u, 0u, 0u, 0u};
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int64_t i = base + h * 64 + lane * 2 + q;
                    if (i < P.n_rec) {
                        const int64_t o = i * B, w = o >> 3;
                        const int sh = (int)(o & 7) * 8;
                        uint64_t r = __ldg(P.rec + w) >> sh;
                        if (sh + 8 * B > 64) r |= __ldg(P.rec + (w < last_word ? w + 1 : last_word)) << (64 - sh);
                        q4[2 * q] = (uint32_t)(r & tmask) | ((uint32_t)((r >> tb) & 1ull) << 31);
                        q4[2 * q + 1] = P.rec_same ? (uint32_t)(r & tmask) : (uint32_t)((r >> (tb + 1)) & tmask);
                        okm |= 1u << (2 * h + q);
                    }
                }
                v[h] = make_uint4(q4[0], q4[1], q4[2], q4[3]);
            }
            return okm;
        }
#pragma unroll
        for (int h = 0; h < CLS_RPT / 2; ++h) {
            const int64_t i = base + h * 64 + lane * 2;
            if (i + 1 < P.n_rec) {
                v[h] = ld_stream_u4(P.rec + i);
                okm |= 3u << (2 * h);
            } else if (i < P.n_rec) {
                const uint2 t = ld_stream_u2(P.rec + i);
                v[h] = make_uint4(t.x, t.y, 0u, 0u);
                okm |= 1u << (2 * h);
            } else {
                v[h] = make_uint4(0u, 0u, 0u, 0u);
            }
        }
        return okm;
    };

    // register ring of three tiles: the loads of the tile after next are issued before this tile is processed
    uint4 v[CLS_RPT / 2], vn[CLS_RPT / 2];
    unsigned okm = 0, okn = 0;
    if (w0 < n_tiles) okm = load_tile(w0, v);
    if (w0 + n_warps < n_tiles) okn = load_tile(w0 + n_warps, vn);
    for (int64_t tile = w0; tile < n_tiles; tile += n_warps) {
        uint4 vnn[CLS_RPT / 2];
        unsigned oknn = 0;
        if (tile + 2 * n_warps < n_tiles) oknn = load_tile(tile + 2 * n_warps, vnn);
        uint64_t keyv[CLS_RPT];
        unsigned offm[CLS_RPT];
        uint32_t ixv[CLS_RPT], jxv[CLS_RPT];
        bool accv[CLS_RPT];
        // all look-ups of the tile first (eight independent shared-memory loads in flight per thread); the second
        // mate of an intra-contig pair -- two thirds of Hi-C pairs -- has the first one's reference and is not looked up
#pragma unroll
        for (int k = 0; k < CLS_RPT; ++k) {
            const uint32_t lo = (k & 1) ? v[k >> 1].z : v[k >> 1].x;
            const uint32_t hi = (k & 1) ? v[k >> 1].w : v[k >> 1].y;
            const bool ok = (okm >> k) & 1u;
            const uint32_t ti = lo & 0x7fffffffu, tj = hi & 0x7fffffffu;
            bool hit_i, hit_j;
            const uint32_t ix = lookup(ti, ok, hit_i);
            uint32_t jx = lookup(tj, ok && tj != ti, hit_j);
            if (tj == ti) {
                jx = ix;
                hit_j = hit_i;
            }
            const bool valid = ok && hit_i && hit_j;            // else excluded: contact_map.py:733-735
            const bool acc = valid && (lo >> 31);               // else poor match: contact_map.py:737-739
            n_ok += ok ? 1u : 0u;
            n_valid += valid ? 1u : 0u;
            n_acc += acc ? 1u : 0u;                             // contact_map.py:796
            ixv[k] = ix;
            jxv[k] = jx;
            accv[k] = acc;
        }
#pragma unroll
        for (int k = 0; k < CLS_RPT; ++k) {
            const uint32_t ix = ixv[k], jx = jxv[k];
            const bool same = ix == jx;
            if (accv[k] && same) {
                if (SMEM_DIAG || ix < dk) atomicAdd(&s_diag[ix], 1u);
                else atomicAdd(&P.diag[ix], 1u);
            }
            const uint32_t a = min(ix, jx), c = max(ix, jx);    // contact_map.py:774-777
            keyv[k] = ((uint64_t)a << P.b) | c;
            offm[k] = __ballot_sync(kFullMask, accv[k] && !same);
        }
        unsigned wtot = 0;
#pragma unroll
        for (int k = 0; k < CLS_RPT; ++k) wtot += __popc(offm[k]);
        if (cnt + wtot > (unsigned)P.cap_w) flush();            // warp-uniform
        unsigned at = cnt;
#pragma unroll
        for (int k = 0; k < CLS_RPT; ++k) {
            if ((offm[k] >> lane) & 1u) s_stage[at + __popc(offm[k] & lt)] = (stage_t)keyv[k];
            at += __popc(offm[k]);
        }
        cnt = at;
#pragma unroll
        for (int h = 0; h < CLS_RPT / 2; ++h) {
            v[h] = vn[h];
            vn[h] = vnn[h];
        }
        okm = okn;
        okn = oknn;
    }
    if (cnt) flush();

    if (dk) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < dk; i += CLS_THREADS) {
            const uint32_t c = s_diag[i];
            if (c) atomicAdd(&P.diag[i], c);
        }
    }
    // counters: warp reduce, then one atomic per warp
    n_ok = warp_sum(n_ok);
    n_valid = warp_sum(n_valid);
    n_acc = warp_sum(n_acc);
    if (lane == 0) {
        if (n_acc) atomicAdd(&P.ctr[C_ACCEPT], (unsigned long long)n_acc);
        if (n_ok - n_valid) atomicAdd(&P.ctr[C_EXCL], (unsigned long long)(n_ok - n_valid));
        if (n_valid - n_acc) atomicAdd(&P.ctr[C_POOR], (unsigned long long)(n_valid - n_acc));
    }
}

template <bool SMEM_DIAG, int SMEM_RANK>
__global__ void __launch_bounds__(CLS_THREADS, 1) k_classify(ClsParams P) {
    extern __shared__ __align__(16) unsigned char smem[];
    // the rank table is only valid when the tid->index map is the dense rank map (checked on device)
    const bool rank_ok = SMEM_RANK && (P.ctr[C_LUT_OK] != 0);
    if (rank_ok) classify_tiles<SMEM_DIAG, SMEM_RANK>(P, smem);
    else classify_tiles<SMEM_DIAG, 0>(P, smem);
}

// an overflowed key buffer must not be sorted: drop the keys, keep the flag (reported by reduce)
__global__ void k_accum_guard(unsigned long long *__restrict__ ctr, int64_t cap) {
    if (ctr[C_OVERFLOW] || (int64_t)ctr[C_NKEYS] > cap) {
        ctr[C_OVERFLOW] = 1;
        ctr[C_NKEYS] = 0;
    }
}

// ---- LSD radix sort --------------------------------------------------------------------
__device__ __forceinline__ void rs_segment(int64_t n, int64_t *lo, int64_t *hi, int64_t *t0, int64_t *t1) {
    const int64_t n_tiles = (n + RS_TILE - 1) / RS_TILE;
    const int64_t tpb = (n_tiles + gridDim.x - 1) / gridDim.x;
    *t0 = min((int64_t)blockIdx.x * tpb, n_tiles);
    *t1 = min(*t0 + tpb, n_tiles);
    *lo = *t0 * RS_TILE;
    *hi = min(n, *t1 * RS_TILE);
}

template <int BITS>
__global__ void __launch_bounds__(RS_THREADS) k_rs_hist(const uint64_t *__restrict__ keys,
                                                        const unsigned long long *__restrict__ d_n, int shift,
                                                        unsigned mask, uint32_t *__restrict__ hist) {
    constexpr int RS_BINS = 1 << BITS;
    __shared__ uint32_t s_h[RS_BINS];
    for (int i = threadIdx.x; i < RS_BINS; i += RS_THREADS) s_h[i] = 0;
    __syncthreads();
    int64_t lo, hi, t0, t1;
    rs_segment((int64_t)*d_n, &lo, &hi, &t0, &t1);
    for (int64_t i = lo + threadIdx.x; i < hi; i += RS_THREADS)
        atomicAdd(&s_h[(unsigned)(keys[i] >> shift) & mask], 1u);
    __syncthreads();
    for (int d = threadIdx.x; d < RS_BINS; d += RS_THREADS) hist[(int64_t)d * gridDim.x + blockIdx.x] = s_h[d];
}

// one CTA per digit: exclusive scan of that digit's per-block counts in place, digit total out.
// The scatter kernel turns the 256 totals into digit bases itself.
__global__ void __launch_bounds__(256) k_rs_scan_digit(uint32_t *__restrict__ hist, int nblk,
                                                      uint32_t *__restrict__ totals) {
    __shared__ uint32_t s_w[33];
    uint32_t *row = hist + (int64_t)blockIdx.x * nblk;
    const int per = (nblk + 255) / 256;
    const int lo = min(nblk, (int)threadIdx.x * per), hi = min(nblk, lo + per);
    uint32_t sum = 0;
    for (int i = lo; i < hi; ++i) sum += row[i];
    uint32_t tot;
    uint32_t ex = block_scan_excl<uint32_t>(sum, s_w, &tot);
    for (int i = lo; i < hi; ++i) {
        const uint32_t v = row[i];
        row[i] = ex;
        ex += v;
    }
    if (threadIdx.x == 0) totals[blockIdx.x] = tot;
}

template <int BITS>
__global__ void __launch_bounds__(RS_THREADS) k_rs_scatter(const uint64_t *__restrict__ in,
                                                           uint64_t *__restrict__ out,
                                                           const unsigned long long *__restrict__ d_n, int shift,
                                                           unsigned mask, const uint32_t *__restrict__ offs,
                                                           const uint32_t *__restrict__ totals) {
    constexpr int RS_BITS = BITS, RS_BINS = 1 << BITS;
    static_assert(RS_BINS <= RS_THREADS, "one thread per digit");
    __shared__ uint32_t s_wcnt[RS_WARPS][RS_BINS + 1];
    __shared__ uint32_t s_off[RS_BINS];
    __shared__ uint32_t s_tot[RS_BINS];
    __shared__ uint32_t s_bin[RS_BINS];
    __shared__ uint32_t s_dst[RS_BINS];         // s_off - s_bin of the current tile: out index = s_dst[d] + q
    __shared__ uint32_t s_scan[33];
    extern __shared__ __align__(16) unsigned char rs_dyn[];
    uint64_t *s_keys = reinterpret_cast<uint64_t *>(rs_dyn);     // RS_TILE keys (32 KB, dynamic)

    const int64_t n = (int64_t)*d_n;
    int64_t lo, hi, t0, t1;
    rs_segment(n, &lo, &hi, &t0, &t1);
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5, lt = lanemask_lt();
    {
        // digit base = exclusive scan of the digit totals; plus this block's offset inside the digit
        const uint32_t v = (threadIdx.x < RS_BINS) ? totals[threadIdx.x] : 0u;
        uint32_t tot;
        const uint32_t ex = block_scan_excl<uint32_t>(v, s_scan, &tot);
        if (threadIdx.x < RS_BINS) s_off[threadIdx.x] = ex + offs[(int64_t)threadIdx.x * gridDim.x + blockIdx.x];
    }
    __syncthreads();

    for (int64_t tile = t0; tile < t1; ++tile) {
        const int64_t base = tile * RS_TILE;
        const int cnt = (int)min((int64_t)RS_TILE, n - base);
        for (int i = threadIdx.x; i < RS_WARPS * (RS_BINS + 1); i += RS_THREADS) (&s_wcnt[0][0])[i] = 0;
        uint64_t key[RS_KPT];
        uint32_t dg[RS_KPT], rk[RS_KPT];
#pragma unroll
        for (int k = 0; k < RS_KPT; ++k) {
            const int idx = warp * (32 * RS_KPT) + k * 32 + lane;     // warp-striped: order == index order
            const bool valid = idx < cnt;
            key[k] = valid ? in[base + idx] : 0ull;
            dg[k] = valid ? ((unsigned)(key[k] >> shift) & mask) : (unsigned)RS_BINS;
        }
        __syncthreads();
        // stable rank inside the warp, one item row at a time.  The peer masks do not depend on the counters, so
        // they are all taken first; then the leader of every match group bumps the warp's digit counter with ONE
        // shared-memory atomic that returns the count of the earlier rows (the rows' atomics are issued back to
        // back: nothing waits for a value until the shuffles below), and the group reads it from the leader.
        unsigned mm[RS_KPT];
#pragma unroll
        for (int k = 0; k < RS_KPT; ++k) {
            // lanes holding the same digit: one ballot per digit bit (match.any is a slow MIO operation here --
            // it was 24 % of this kernel's stall samples); invalid lanes (digit RS_BINS) form their own group
            const bool valid = dg[k] < (unsigned)RS_BINS;
            unsigned m = __ballot_sync(kFullMask, valid);
            if (!valid) m = ~m;
#pragma unroll
            for (int b = 0; b < RS_BITS; ++b) {
                const bool bit = (dg[k] >> b) & 1u;
                const unsigned bal = __ballot_sync(kFullMask, bit);
                m &= bit ? bal : ~bal;
            }
            mm[k] = m;
        }
#pragma unroll
        for (int k = 0; k < RS_KPT; ++k) {
            rk[k] = 0;
            if ((int)lane == __ffs(mm[k]) - 1) rk[k] = atomicAdd(&s_wcnt[warp][dg[k]], (uint32_t)__popc(mm[k]));
            __syncwarp();                          // row k's additions are ordered before row k + 1's
        }
#pragma unroll
        for (int k = 0; k < RS_KPT; ++k)
            rk[k] = __shfl_sync(kFullMask, rk[k], __ffs(mm[k]) - 1) + __popc(mm[k] & lt);
        __syncthreads();
        // per digit: exclusive scan over warps, tile total
        if (threadIdx.x < RS_BINS) {
            uint32_t run = 0;
#pragma unroll
            for (int w = 0; w < RS_WARPS; ++w) {
                const uint32_t c = s_wcnt[w][threadIdx.x];
                s_wcnt[w][threadIdx.x] = run;
                run += c;
            }
            s_tot[threadIdx.x] = run;
        }
        __syncthreads();
        {
            const uint32_t v = (threadIdx.x < RS_BINS) ? s_tot[threadIdx.x] : 0u;
            uint32_t tot;
            const uint32_t ex = block_scan_excl<uint32_t>(v, s_scan, &tot);
            if (threadIdx.x < RS_BINS) {
                // digit d's keys of this tile go to out[s_off[d] ...]; thread d alone touches s_off[d], so it moves
                // on to the next tile here (the write-out below reads s_dst): no barrier at the end of the tile
                s_bin[threadIdx.x] = ex;
                s_dst[threadIdx.x] = s_off[threadIdx.x] - ex;            // (mod 2^32, undone by + q below)
                s_off[threadIdx.x] += v;
            }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < RS_KPT; ++k)
            if (dg[k] < (unsigned)RS_BINS) s_keys[s_bin[dg[k]] + s_wcnt[warp][dg[k]] + rk[k]] = key[k];
        __syncthreads();
        for (int q = threadIdx.x; q < cnt; q += RS_THREADS) {
            const uint64_t kk = s_keys[q];
            const unsigned d = (unsigned)(kk >> shift) & mask;
            out[(int64_t)(uint32_t)(s_dst[d] + (uint32_t)q)] = kk;
        }
        // the next tile's first writes to s_wcnt / s_keys / s_tot / s_bin / s_dst all lie behind its own barriers;
        // s_wcnt (zeroed at the top) was last read before the barrier above
    }
}

// sort keys on bits [bit_lo, bit_hi); returns the index (0=a,1=b) of the buffer with the result
// Digits are as wide as it takes to sort `bits` bits in the fewest passes of at most 9 bits (36 key bits: 4 x 9
// instead of 5 x 8; 18 column bits: 2 x 9 instead of 3 x 8); where 8-bit digits need no more passes (32 bits: 4 x 8)
// the lighter 256-bin kernels run.
static int radix_passes(int bits) { return bits <= 0 ? 0 : (bits + RS_BITS - 1) / RS_BITS; }

// bits per digit of radix_sort over `bits` bits (the last pass may take fewer); above 8 the 512-bin kernels run
static int radix_digit(int bits) {
    const int passes = radix_passes(bits);
    return passes > 0 ? (bits + passes - 1) / passes : 0;
}

// which buffer (0 = a, 1 = b) holds the result of radix_sort over these bits: the parity of the pass count
static int radix_where(int bit_lo, int bit_hi) { return radix_passes(bit_hi - bit_lo) & 1; }

// once per process, outside any graph capture
static int radix_init() {
    static bool attr_done = false;
    if (!attr_done) {
        B3C_CUDA(cudaFuncSetAttribute(k_rs_scatter<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, RS_TILE * 8));
        B3C_CUDA(cudaFuncSetAttribute(k_rs_scatter<9>, cudaFuncAttributeMaxDynamicSharedMemorySize, RS_TILE * 8));
        attr_done = true;
    }
    return B3C_OK;
}

static int radix_sort(uint64_t *a, uint64_t *b, const unsigned long long *d_n, int bit_lo, int bit_hi,
                      uint32_t *d_hist, cudaStream_t s, int *where) {
    const int bits = bit_hi - bit_lo, passes = radix_passes(bits);
    const bool wide = passes > 0 && passes * 8 < bits;           // 8-bit digits would need another pass
    const int digit = radix_digit(bits);
    int cur = 0;
    for (int shift = bit_lo; shift < bit_hi; shift += digit) {
        const int w = (bit_hi - shift) < digit ? (bit_hi - shift) : digit;
        const unsigned mask = (1u << w) - 1u;
        const int bins = wide ? 512 : 256;
        const uint64_t *src = cur ? b : a;
        uint64_t *dst = cur ? a : b;
        uint32_t *d_totals = d_hist + (int64_t)bins * RS_BLOCKS;
        if (wide) k_rs_hist<9><<<RS_BLOCKS, RS_THREADS, 0, s>>>(src, d_n, shift, mask, d_hist);
        else k_rs_hist<8><<<RS_BLOCKS, RS_THREADS, 0, s>>>(src, d_n, shift, mask, d_hist);
        B3C_LAUNCH_CHECK();
        k_rs_scan_digit<<<bins, 256, 0, s>>>(d_hist, RS_BLOCKS, d_totals);
        B3C_LAUNCH_CHECK();
        if (wide) k_rs_scatter<9><<<RS_BLOCKS, RS_THREADS, RS_TILE * 8, s>>>(src, dst, d_n, shift, mask, d_hist, d_totals);
        else k_rs_scatter<8><<<RS_BLOCKS, RS_THREADS, RS_TILE * 8, s>>>(src, dst, d_n, shift, mask, d_hist, d_totals);
        B3C_LAUNCH_CHECK();
        cur ^= 1;
    }
    *where = cur;
    return B3C_OK;
}

// ---- composite of the mirror half ------------------------------------------------------------
// The lower half of the symmetric matrix is the upper half transposed: entry (i, j, c) of the unique list becomes
// (row j, column i, count c).  It is produced by a stable sort on the column bits of a COMPOSITE that carries its own
// payload -- j in the top b bits, then i, then the count in the remaining cbits = min(32, 64 - 2b) bits -- so the emit
// kernel streams the sorted composites instead of gathering i and c through an entry id (at C3 those scattered 8- and
// 4-byte gathers moved 6 GB through DRAM for 0.44 GB of payload).  A count that does not fit (>= 2^cbits - 1) is stored
// as the all-ones escape and looked up exactly by bisection in the sorted unique keys.
__host__ __device__ __forceinline__ int comp_cbits(int b) { return 64 - 2 * b < 32 ? 64 - 2 * b : 32; }

// ---- run-length reduce ----------------------------------------------------------------------
__global__ void __launch_bounds__(RS_THREADS) k_rle_count(const uint64_t *__restrict__ keys,
                                                          const unsigned long long *__restrict__ d_n,
                                                          int64_t *__restrict__ heads) {
    __shared__ unsigned s_c;
    if (threadIdx.x == 0) s_c = 0;
    __syncthreads();
    int64_t lo, hi, t0, t1;
    rs_segment((int64_t)*d_n, &lo, &hi, &t0, &t1);
    unsigned c = 0;
    for (int64_t i = lo + threadIdx.x; i < hi; i += RS_THREADS) c += (i == 0 || keys[i] != keys[i - 1]) ? 1u : 0u;
    c = warp_sum(c);
    if (lane_id() == 0 && c) atomicAdd(&s_c, c);
    __syncthreads();
    if (threadIdx.x == 0) heads[blockIdx.x] = s_c;
}

__global__ void __launch_bounds__(RS_THREADS) k_rle_write(const uint64_t *__restrict__ keys,
                                                          const unsigned long long *__restrict__ d_n,
                                                          const int64_t *__restrict__ heads_ex,
                                                          uint64_t *__restrict__ uniq, uint32_t *__restrict__ pos) {
    __shared__ uint32_t s_w[33];
    int64_t lo, hi, t0, t1;
    rs_segment((int64_t)*d_n, &lo, &hi, &t0, &t1);
    int64_t run = heads_ex[blockIdx.x];
    for (int64_t base = lo; base < hi; base += RS_THREADS) {
        const int64_t i = base + threadIdx.x;
        uint64_t k = 0;
        uint32_t h = 0;
        if (i < hi) {
            k = keys[i];
            h = (i == 0 || k != keys[i - 1]) ? 1u : 0u;
        }
        uint32_t tot;
        const uint32_t ex = block_scan_excl<uint32_t>(h, s_w, &tot);
        if (h) {
            uniq[run + ex] = k;
            pos[run + ex] = (uint32_t)i;
        }
        run += tot;
    }
}

__global__ void k_rle_finish(const int64_t *__restrict__ heads_ex, int nblk, const unsigned long long *d_n,
                             uint32_t *__restrict__ pos, unsigned long long *__restrict__ ctr) {
    const int64_t nnz = heads_ex[nblk];
    ctr[C_NNZ_UO] = (unsigned long long)nnz;
    pos[nnz] = (uint32_t)*d_n;
}

__global__ void k_rle_counts(const uint32_t *__restrict__ pos, const unsigned long long *__restrict__ ctr,
                             uint32_t *__restrict__ cnt, int b, const uint64_t *__restrict__ uniq,
                             uint64_t *__restrict__ comp) {
    const int64_t nnz = (int64_t)ctr[C_NNZ_UO];
    const uint64_t jmask = (1ull << b) - 1ull;
    unsigned long long w = 0;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t c = pos[e + 1] - pos[e];
        cnt[e] = c;
        w += c;
        const int cbits = comp_cbits(b);
        const uint64_t cmask = cbits >= 64 ? ~0ull : ((1ull << cbits) - 1ull);
        const uint64_t k = uniq[e];
        const uint64_t cc = (uint64_t)c < cmask ? (uint64_t)c : cmask;      // all ones: escape, looked up exactly
        comp[e] = ((k & jmask) << (b + cbits)) | ((k >> b) << cbits) | cc;  // (column j, row i, count)
    }
    w = warp_sum(w);
    if (lane_id() == 0 && w) atomicAdd((unsigned long long *)&ctr[C_WEIGHT], 2ull * w);   // mirrored entries (Q7)
}

__global__ void k_diag_stats(const uint32_t *__restrict__ diag, int32_t n, unsigned long long *__restrict__ ctr) {
    unsigned long long nz = 0, w = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t c = diag[i];
        nz += c ? 1ull : 0ull;
        w += c;
    }
    nz = warp_sum(nz);
    w = warp_sum(w);
    if (lane_id() == 0) {
        if (nz) atomicAdd(&ctr[C_NNZ_DIAG], nz);
        if (w) atomicAdd(&ctr[C_WEIGHT], w);
    }
}

// ptr[r] = first entry whose row >= r, ptr[n_seq] = n; rows come from sorted keys >> shift
__global__ void k_row_ptr(const uint64_t *__restrict__ keys, const unsigned long long *__restrict__ d_n, int shift,
                          int32_t n_seq, int64_t *__restrict__ ptr) {
    const int64_t n = (int64_t)*d_n;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t e = gid; e < n; e += stride) {
        if (e == 0) continue;                          // the rows up to the first key's are filled in parallel below
        const int64_t r = (int64_t)(keys[e] >> shift);
        const int64_t rp = (int64_t)(keys[e - 1] >> shift);
        for (int64_t q = rp + 1; q <= r; ++q) ptr[q] = e;
    }
    // Leading and trailing rows without keys.  A row block of a sharded run starts at row_lo: one thread walking
    // there alone cost the last of 8 ranks ~1 ms at C3 and ~4 ms at C4 -- the whole grid does it instead.
    const int64_t rf = n > 0 ? (int64_t)(keys[0] >> shift) : -1;
    for (int64_t q = gid; q <= rf; q += stride) ptr[q] = 0;
    const int64_t rl = n > 0 ? (int64_t)(keys[n - 1] >> shift) : -1;
    for (int64_t q = rl + 1 + gid; q <= n_seq; q += stride) ptr[q] = n;
}

__global__ void k_row_len(const int64_t *__restrict__ up, const int64_t *__restrict__ lo,
                          const uint32_t *__restrict__ diag, int32_t n, int64_t *__restrict__ len_f,
                          int64_t *__restrict__ len_u) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
        const int64_t u = up[r + 1] - up[r], l = lo[r + 1] - lo[r], d = diag[r] ? 1 : 0;
        len_f[r] = u + l + d;
        len_u[r] = u + d;
    }
}

__global__ void k_emit(int symmetric, int b, int32_t n_seq, const unsigned long long *__restrict__ ctr,
                       const uint64_t *__restrict__ uniq, const uint32_t *__restrict__ cnt,
                       const uint64_t *__restrict__ comp, const uint32_t *__restrict__ diag,
                       const int64_t *__restrict__ up, const int64_t *__restrict__ lo,
                       const int64_t *__restrict__ indptr, int32_t *__restrict__ indices,
                       uint32_t *__restrict__ counts) {
    const int64_t nnz = (int64_t)ctr[C_NNZ_UO];
    const uint64_t jmask = (1ull << b) - 1ull;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    // upper half: entry e sits after the row's lower half and diagonal
    for (int64_t e = gid; e < nnz; e += stride) {
        const uint64_t k = uniq[e];
        const int64_t i = (int64_t)(k >> b);
        const int64_t lower = symmetric ? (lo[i + 1] - lo[i]) : 0;
        const int64_t d = indptr[i] + lower + (diag[i] ? 1 : 0) + (e - up[i]);
        indices[d] = (int32_t)(k & jmask);
        counts[d] = cnt[e];
    }
    // diagonal
    for (int64_t r = gid; r < n_seq; r += stride) {
        const uint32_t c = diag[r];
        if (c) {
            const int64_t d = indptr[r] + (symmetric ? (lo[r + 1] - lo[r]) : 0);
            indices[d] = (int32_t)r;
            counts[d] = c;
        }
    }
    // lower half (mirror): composite t is sorted by (column j, row i) and carries the count
    if (symmetric) {
        const int cbits = comp_cbits(b);
        const uint64_t cmask = (1ull << cbits) - 1ull;
        for (int64_t t = gid; t < nnz; t += stride) {
            const uint64_t c = comp[t];
            const int64_t j = (int64_t)(c >> (b + cbits));
            const uint64_t i = (c >> cbits) & jmask;
            uint32_t cv = (uint32_t)(c & cmask);
            if ((c & cmask) == cmask) {                 // escape: the exact count sits beside the unique key (i, j)
                const uint64_t key = (i << b) | (uint64_t)j;
                int64_t a = 0, z = nnz;
                while (a < z) {
                    const int64_t mid = (a + z) >> 1;
                    if (uniq[mid] < key) a = mid + 1;
                    else z = mid;
                }
                cv = cnt[a];
            }
            const int64_t d = indptr[j] + (t - lo[j]);
            indices[d] = (int32_t)i;
            counts[d] = cv;
        }
    }
}

// ==== sharded accumulation (multi-GPU): route keys to the rank that owns their row ================
// Canonical key (i<j) -> two directed keys: (i,j) for the owner of row i, (j,i) for the owner of
// row j.  Each rank then sorts and run-length reduces the directed keys of its own row block, which
// yields the full symmetric rows of that block directly (no mirror sort).
constexpr int ROUTE_MAX_RANKS = 64;

__device__ __forceinline__ int owner_of(int32_t row, const int32_t *s_splits, int G) {
    int g = 0;
    while (g + 1 < G && row >= s_splits[g + 1]) ++g;
    return g;
}

// rowcnt[r] += number of directed keys with row r (int64 so the host side can all-reduce it)
__global__ void k_row_hist(const uint64_t *__restrict__ keys, const unsigned long long *__restrict__ d_n, int b,
                           unsigned long long *__restrict__ rowcnt) {
    const int64_t n = (int64_t)*d_n;
    const uint64_t jmask = (1ull << b) - 1ull;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t k = keys[e];
        atomicAdd(&rowcnt[k >> b], 1ull);
        atomicAdd(&rowcnt[k & jmask], 1ull);
    }
}

__global__ void __launch_bounds__(256) k_route_count(const uint64_t *__restrict__ keys,
                                                     const unsigned long long *__restrict__ d_n, int b,
                                                     const int32_t *__restrict__ splits, int G,
                                                     unsigned long long *__restrict__ cnt) {
    __shared__ int32_t s_splits[ROUTE_MAX_RANKS + 1];
    __shared__ unsigned s_cnt[ROUTE_MAX_RANKS];
    if (threadIdx.x <= (unsigned)G) s_splits[threadIdx.x] = splits[threadIdx.x];
    if (threadIdx.x < (unsigned)G) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const int64_t n = (int64_t)*d_n;
    const uint64_t jmask = (1ull << b) - 1ull;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t k = keys[e];
        atomicAdd(&s_cnt[owner_of((int32_t)(k >> b), s_splits, G)], 1u);
        atomicAdd(&s_cnt[owner_of((int32_t)(k & jmask), s_splits, G)], 1u);
    }
    __syncthreads();
    if (threadIdx.x < (unsigned)G && s_cnt[threadIdx.x]) atomicAdd(&cnt[threadIdx.x], (unsigned long long)s_cnt[threadIdx.x]);
}

// base[g] = exclusive scan of cnt; cursor[g] starts at base[g]
__global__ void k_route_bases(const unsigned long long *__restrict__ cnt, int G, unsigned long long *__restrict__ base,
                              unsigned long long *__restrict__ cursor) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        unsigned long long run = 0;
        for (int g = 0; g < G; ++g) {
            base[g] = run;
            cursor[g] = run;
            run += cnt[g];
        }
        base[G] = run;
    }
}

__global__ void __launch_bounds__(256) k_route_scatter(const uint64_t *__restrict__ keys,
                                                       const unsigned long long *__restrict__ d_n, int b,
                                                       const int32_t *__restrict__ splits, int G,
                                                       unsigned long long *__restrict__ cursor,
                                                       uint64_t *__restrict__ out) {
    __shared__ int32_t s_splits[ROUTE_MAX_RANKS + 1];
    __shared__ unsigned s_cnt[ROUTE_MAX_RANKS];
    __shared__ unsigned long long s_base[ROUTE_MAX_RANKS];
    if (threadIdx.x <= (unsigned)G) s_splits[threadIdx.x] = splits[threadIdx.x];
    __syncthreads();
    const int64_t n = (int64_t)*d_n;
    const uint64_t jmask = (1ull << b) - 1ull;
    const int64_t per_block = 256 * 8;
    for (int64_t base = (int64_t)blockIdx.x * per_block; base < n; base += (int64_t)gridDim.x * per_block) {
        if (threadIdx.x < (unsigned)G) s_cnt[threadIdx.x] = 0;
        __syncthreads();
        uint64_t dk[16];
        int own[16];
        unsigned slot[16];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int64_t e = base + q * 256 + threadIdx.x;
            if (e < n) {
                const uint64_t k = keys[e];
                const uint64_t i = k >> b, j = k & jmask;
                dk[2 * q] = k;
                dk[2 * q + 1] = (j << b) | i;
                own[2 * q] = owner_of((int32_t)i, s_splits, G);
                own[2 * q + 1] = owner_of((int32_t)j, s_splits, G);
                slot[2 * q] = atomicAdd(&s_cnt[own[2 * q]], 1u);
                slot[2 * q + 1] = atomicAdd(&s_cnt[own[2 * q + 1]], 1u);
            } else {
                own[2 * q] = own[2 * q + 1] = -1;
            }
        }
        __syncthreads();
        if (threadIdx.x < (unsigned)G && s_cnt[threadIdx.x])
            s_base[threadIdx.x] = atomicAdd(&cursor[threadIdx.x], (unsigned long long)s_cnt[threadIdx.x]);
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 16; ++q)
            if (own[q] >= 0) out[s_base[own[q]] + slot[q]] = dk[q];
        __syncthreads();
    }
}

// row block emit: unique directed keys (row in [row_lo,row_hi), col != row) + diagonal -> local CSR.
// ptr[] is the row pointer over GLOBAL rows (k_row_ptr); indptr is local (row_hi - row_lo + 1).
__global__ void k_block_row_len(const int64_t *__restrict__ ptr, const uint32_t *__restrict__ diag, int32_t row_lo,
                                int32_t n_local, int64_t *__restrict__ len) {
    for (int64_t lr = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; lr < n_local; lr += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = row_lo + lr;
        len[lr] = (ptr[r + 1] - ptr[r]) + (diag[r] ? 1 : 0);
    }
}

// One thread per entry of the block (the key holds its row), then one per row for the diagonal, placed by bisection
// among the row's sorted columns: a warp-per-row walk left the longest row of a heavy-tailed community to one warp
// (C4 on 8 GPUs: 2.2 ms on the rank that held it against 1.1 ms elsewhere).
__global__ void __launch_bounds__(256) k_emit_block(int b, int32_t row_lo, int32_t n_local,
                                                    const uint64_t *__restrict__ uniq, const uint32_t *__restrict__ cnt,
                                                    const uint32_t *__restrict__ diag, const int64_t *__restrict__ ptr,
                                                    const int64_t *__restrict__ indptr, int32_t *__restrict__ indices,
                                                    uint32_t *__restrict__ counts) {
    const uint64_t jmask = (1ull << b) - 1ull;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t e_lo = ptr[row_lo], e_hi = ptr[row_lo + n_local];
    for (int64_t e = e_lo + gid; e < e_hi; e += stride) {
        const uint64_t k = uniq[e];
        const int64_t r = (int64_t)(k >> b);
        const int32_t c = (int32_t)(k & jmask);
        const int64_t dst = indptr[r - row_lo] + (e - ptr[r]) + ((c >= (int32_t)r && diag[r]) ? 1 : 0);
        indices[dst] = c;
        counts[dst] = cnt[e];
    }
    for (int64_t lr = gid; lr < n_local; lr += stride) {
        const int64_t r = row_lo + lr;
        const uint32_t d = diag[r];
        if (!d) continue;
        int64_t a = ptr[r], z = ptr[r + 1];
        const int64_t first = a;
        while (a < z) {                                 // entries of the row with column < r
            const int64_t mid = (a + z) >> 1;
            if ((int64_t)(uniq[mid] & jmask) < r) a = mid + 1;
            else z = mid;
        }
        indices[indptr[lr] + (a - first)] = (int32_t)r;
        counts[indptr[lr] + (a - first)] = d;
    }
}


// ---- peer exchange arena (multi-GPU, one process per GPU of a node) ------------------------------------
// Every rank owns one arena, allocated with b3c_peer_alloc and mapped by all other ranks over NVLink
// (CUDA IPC).  Ranks write into each other's arenas directly from kernels -- routed keys, mask and x
// slices, small reduction operands -- and synchronise with flag barriers kept in the same arenas, so
// the data path of the sharded accumulation has no collective-library call and no host round trip.
constexpr int XA_MAX_RANKS = 8;
constexpr int XA_SCAL = 8;                       // doubles per small all-reduce
constexpr int XA_CHUNK = 1024;                   // rows per weight chunk = KR's reduction chunk (row-block alignment)
constexpr int XA_MAX_CHUNKS = 4096;              // weight chunks the split kernel keeps in shared memory

struct XaLayout {
    int64_t o_flag, o_ctl, o_scal, o_cw, o_cnt3, o_diag, o_mask, o_x, o_keys, total;
    int32_t n_chunks;
};
static XaLayout xa_layout(int32_t n_seq, int64_t key_cap) {
    XaLayout X;
    Carver c;
    X.n_chunks = (int32_t)ceil_div(n_seq, XA_CHUNK);
    X.o_flag = c.take(XA_MAX_RANKS * 8);
    X.o_ctl = c.take(4 * 8);                                     // [0] keys received, [1] overflow, [2] time-out
    X.o_scal = c.take(2 * XA_MAX_RANKS * XA_SCAL * 8);           // two sets, alternated by barrier epoch
    X.o_cw = c.take((int64_t)XA_MAX_RANKS * X.n_chunks * 8);
    X.o_cnt3 = c.take(XA_MAX_RANKS * 4 * 8);
    X.o_diag = c.take((int64_t)n_seq * 4);
    X.o_mask = c.take((int64_t)n_seq);
    X.o_x = c.take((int64_t)n_seq * 8);
    X.o_keys = c.take((key_cap > 0 ? key_cap : 1) * 8);
    X.total = c.cur;
    return X;
}

struct Peers {
    char *a[XA_MAX_RANKS];
};

// Flag barrier between the ranks' streams: everything this rank enqueued before it is complete (stream
// order), thread g tells rank g "rank `rank` reached `epoch`" and waits until rank g has told us the same.
// A rank that never arrives would hang the node, so the wait gives up after the peer time-out (60 s unless
// B3C_OPT_PEER_TIMEOUT_MS says otherwise: ordinary rank skew -- a slower BAM shard, an allocator stall -- must not
// trip it) and raises the arena's time-out word, reported by the next call that synchronises; the results of a
// run that timed out are invalid.
__global__ void k_peer_barrier(Peers P, int rank, int G, unsigned long long epoch, int64_t o_flag, int64_t o_ctl,
                               long long timeout) {
    const int g = threadIdx.x;
    if (g >= G) return;
    __threadfence_system();
    unsigned long long *theirs = (unsigned long long *)(P.a[g] + o_flag) + rank;
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(theirs), "l"(epoch) : "memory");
    const unsigned long long *mine = (const unsigned long long *)(P.a[rank] + o_flag) + g;
    const long long t0 = clock64();
    unsigned long long seen;
    do {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(mine) : "memory");
        if (seen < epoch && clock64() - t0 > timeout) {
            ((unsigned long long *)(P.a[rank] + o_ctl))[2] = 1ull;
            break;
        }
    } while (seen < epoch);
}

// copy `bytes` (a multiple of 1; 16-byte aligned fast path) from src into every rank's arena at `offset`
__global__ void k_peer_put(Peers P, int G, int64_t offset, const unsigned char *__restrict__ src, int64_t bytes) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool vec = ((offset | (int64_t)(uintptr_t)src) & 15) == 0;
    const int64_t nv = vec ? bytes / 16 : 0;
    for (int g = 0; g < G; ++g) {
        unsigned char *dst = (unsigned char *)(P.a[g] + offset);
        for (int64_t i = gid; i < nv; i += stride) ((uint4 *)dst)[i] = ((const uint4 *)src)[i];
        for (int64_t i = nv * 16 + gid; i < bytes; i += stride) dst[i] = src[i];
    }
}

// all-reduce of up to XA_SCAL doubles: put this rank's values into slot `rank` of every arena, flag barrier,
// reduce the G slots in rank order (the same order on every rank: bit-identical results).  One CTA.
__global__ void k_peer_allreduce(Peers P, int rank, int G, unsigned long long epoch, int op, double *__restrict__ val,
                                 int count, int64_t o_flag, int64_t o_ctl, int64_t o_scal, long long timeout) {
    const int64_t set = o_scal + (int64_t)(epoch & 1ull) * XA_MAX_RANKS * XA_SCAL * 8;
    const int t = threadIdx.x;
    if (t < G * count) {
        const int g = t / count, i = t % count;
        ((double *)(P.a[g] + set))[rank * XA_SCAL + i] = val[i];
    }
    __syncthreads();
    if (t < G) {
        __threadfence_system();
        unsigned long long *theirs = (unsigned long long *)(P.a[t] + o_flag) + rank;
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(theirs), "l"(epoch) : "memory");
        const unsigned long long *mine = (const unsigned long long *)(P.a[rank] + o_flag) + t;
        const long long t0 = clock64();
        unsigned long long seen;
        do {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(mine) : "memory");
            if (seen < epoch && clock64() - t0 > timeout) {
                ((unsigned long long *)(P.a[rank] + o_ctl))[2] = 1ull;
                break;
            }
        } while (seen < epoch);
    }
    __syncthreads();
    if (t < count) {
        const volatile double *slots = (const volatile double *)(P.a[rank] + set);
        double r = slots[t];
        for (int g = 1; g < G; ++g) {
            const double v = slots[g * XA_SCAL + t];
            r = op == 0 ? r + v : fmax(r, v);
        }
        val[t] = r;
    }
}

// cw[c] += directed keys whose row lies in 1024-row chunk c (both directions of every canonical key)
__global__ void __launch_bounds__(256) k_chunk_weights(const uint64_t *__restrict__ keys,
                                                       const unsigned long long *__restrict__ d_n, int b, int n_chunks,
                                                       unsigned long long *__restrict__ cw) {
    extern __shared__ unsigned s_cw[];
    const bool sm = n_chunks <= XA_MAX_CHUNKS;
    if (sm) {
        for (int i = threadIdx.x; i < n_chunks; i += blockDim.x) s_cw[i] = 0;
        __syncthreads();
    }
    const int64_t n = (int64_t)*d_n;
    const uint64_t jmask = (1ull << b) - 1ull;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t k = keys[e];
        const int ci = (int)((k >> b) / XA_CHUNK), cj = (int)((k & jmask) / XA_CHUNK);
        if (sm) {
            atomicAdd(&s_cw[ci], 1u);
            atomicAdd(&s_cw[cj], 1u);
        } else {
            atomicAdd(&cw[ci], 1ull);
            atomicAdd(&cw[cj], 1ull);
        }
    }
    if (sm) {
        __syncthreads();
        for (int i = threadIdx.x; i < n_chunks; i += blockDim.x)
            if (s_cw[i]) atomicAdd(&cw[i], (unsigned long long)s_cw[i]);
    }
}

// this rank's pair counters into slot `rank` of every arena
__global__ void k_publish_counters(Peers P, int rank, int G, const unsigned long long *__restrict__ ctr, int64_t o_cnt3) {
    const int t = threadIdx.x;
    if (t < G * 3) {
        const int g = t / 3, i = t % 3;
        ((unsigned long long *)(P.a[g] + o_cnt3))[rank * 4 + i] = ctr[C_ACCEPT + i];
    }
}

// Row splits from the summed chunk weights: G contiguous row ranges of about equal weight (directed keys
// + one diagonal entry per row), cut at chunk boundaries; splits[G] = n_seq.  Every rank computes the same
// table from the same numbers.  One CTA.
__global__ void __launch_bounds__(1024) k_shard_splits(Peers P, int rank, int G, int32_t n_seq, int n_chunks,
                                                       int64_t o_cw, int32_t *__restrict__ splits) {
    __shared__ long long s_cum[XA_MAX_CHUNKS];
    const unsigned long long *cw = (const unsigned long long *)(P.a[rank] + o_cw);
    for (int c = threadIdx.x; c < n_chunks; c += blockDim.x) {
        long long w = 0;
        for (int g = 0; g < G; ++g) w += (long long)cw[(int64_t)g * n_chunks + c];
        const int64_t rows = (int64_t)n_seq - (int64_t)c * XA_CHUNK;
        s_cum[c] = w + (rows < XA_CHUNK ? rows : XA_CHUNK);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        long long run = 0;
        for (int c = 0; c < n_chunks; ++c) {
            run += s_cum[c];
            s_cum[c] = run;                                  // inclusive
        }
        const long long total = run;
        const int full = n_seq / XA_CHUNK;                   // cuts lie on whole-chunk boundaries below n_seq
        int prev = 0, c = 0;
        splits[0] = 0;
        for (int k = 1; k < G; ++k) {
            const long long target = total * k / G;
            while (c < n_chunks && s_cum[c] < target) ++c;   // first chunk whose inclusive sum reaches the target
            int bnd = c;                                     // boundary before chunk c ...
            if (c < n_chunks) {
                const long long before = c > 0 ? s_cum[c - 1] : 0;
                if (s_cum[c] - target <= target - before) bnd = c + 1;      // ... or after it, whichever is nearer
            }
            if (bnd > full) bnd = full;
            if (bnd < prev) bnd = prev;
            prev = bnd;
            splits[k] = bnd * XA_CHUNK;
        }
        splits[G] = n_seq;
    }
}

// Route + scatter over NVLink: every canonical key (i<j) becomes the directed keys (i,j) and (j,i); each goes
// straight into the receive buffer of the rank that owns its row.  Per tile the keys are grouped by owner in
// shared memory, one system-scope atomic per owner reserves the range in that rank's buffer, and the tile is
// written out in owner-contiguous, coalesced runs.
constexpr int RT_THREADS = 256;
constexpr int RT_KPT = 8;
constexpr int RT_TILE = RT_THREADS * RT_KPT;
__global__ void __launch_bounds__(RT_THREADS) k_route_peer(const uint64_t *__restrict__ keys,
                                                           const unsigned long long *__restrict__ d_n, int b,
                                                           const int32_t *__restrict__ splits, Peers P, int G,
                                                           int64_t o_ctl, int64_t o_keys, int64_t cap) {
    __shared__ int32_t s_splits[XA_MAX_RANKS + 1];
    __shared__ unsigned s_cnt[XA_MAX_RANKS], s_off[XA_MAX_RANKS + 1];
    __shared__ unsigned long long s_base[XA_MAX_RANKS];
    __shared__ uint64_t s_stage[2 * RT_TILE];
    if (threadIdx.x <= (unsigned)G) s_splits[threadIdx.x] = splits[threadIdx.x];
    __syncthreads();
    const int64_t n = (int64_t)*d_n;
    const uint64_t jmask = (1ull << b) - 1ull;
    for (int64_t base = (int64_t)blockIdx.x * RT_TILE; base < n; base += (int64_t)gridDim.x * RT_TILE) {
        if (threadIdx.x < (unsigned)G) s_cnt[threadIdx.x] = 0;
        __syncthreads();
        uint64_t dk[2 * RT_KPT];
        int own[2 * RT_KPT];
        unsigned slot[2 * RT_KPT];
#pragma unroll
        for (int q = 0; q < RT_KPT; ++q) {
            const int64_t e = base + q * RT_THREADS + threadIdx.x;
            if (e < n) {
                const uint64_t k = keys[e];
                const uint64_t i = k >> b, j = k & jmask;
                dk[2 * q] = k;
                dk[2 * q + 1] = (j << b) | i;
                own[2 * q] = owner_of((int32_t)i, s_splits, G);
                own[2 * q + 1] = owner_of((int32_t)j, s_splits, G);
                slot[2 * q] = atomicAdd(&s_cnt[own[2 * q]], 1u);
                slot[2 * q + 1] = atomicAdd(&s_cnt[own[2 * q + 1]], 1u);
            } else {
                own[2 * q] = own[2 * q + 1] = -1;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned run = 0;
            for (int g = 0; g < G; ++g) {
                s_off[g] = run;
                run += s_cnt[g];
            }
            s_off[G] = run;
        }
        if (threadIdx.x < (unsigned)G && s_cnt[threadIdx.x]) {
            unsigned long long *ctl = (unsigned long long *)(P.a[threadIdx.x] + o_ctl);
            const unsigned long long at = atomicAdd_system(&ctl[0], (unsigned long long)s_cnt[threadIdx.x]);
            if ((int64_t)(at + s_cnt[threadIdx.x]) > cap) {
                ctl[1] = 1ull;                               // receive buffer overflow: drop, the owner reports it
                s_base[threadIdx.x] = ~0ull;
            } else {
                s_base[threadIdx.x] = at;
            }
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 2 * RT_KPT; ++q)
            if (own[q] >= 0) s_stage[s_off[own[q]] + slot[q]] = dk[q];
        __syncthreads();
        const unsigned total = s_off[G];
        for (unsigned i = threadIdx.x; i < total; i += RT_THREADS) {
            int g = 0;
            while (i >= s_off[g + 1]) ++g;
            const unsigned long long at = s_base[g];
            if (at != ~0ull) ((uint64_t *)(P.a[g] + o_keys))[at + (i - s_off[g])] = s_stage[i];
        }
        __syncthreads();
    }
}

// diag[r] = sum over ranks of their diagonal histograms, for this rank's rows (peer reads)
__global__ void k_diag_gather(Peers P, int G, int32_t row_lo, int32_t row_hi, int64_t o_diag, uint32_t *__restrict__ diag) {
    for (int64_t r = row_lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < row_hi; r += (int64_t)gridDim.x * blockDim.x) {
        uint32_t s = 0;
        for (int g = 0; g < G; ++g) s += ((const uint32_t *)(P.a[g] + o_diag))[r];
        diag[r] = s;
    }
}

// received-key count -> the sort's counter; summed pair counters; flags
__global__ void k_shard_collect(Peers P, int rank, int G, int64_t o_ctl, int64_t o_cnt3, int64_t cap,
                                unsigned long long *__restrict__ ctr, unsigned long long *__restrict__ out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const unsigned long long *ctl = (const unsigned long long *)(P.a[rank] + o_ctl);
    const unsigned long long *c3 = (const unsigned long long *)(P.a[rank] + o_cnt3);
    const bool bad = ctl[1] != 0 || (int64_t)ctl[0] > cap;
    ctr[C_NKEYS] = bad ? 0ull : ctl[0];
    ctr[C_NNZ_UO] = ctr[C_NNZ_DIAG] = ctr[C_WEIGHT] = 0ull;
    out[0] = ctl[0];
    out[1] = bad ? 1ull : 0ull;
    out[2] = ctl[2];
    for (int i = 0; i < 3; ++i) {
        unsigned long long s = 0;
        for (int g = 0; g < G; ++g) s += c3[g * 4 + i];
        out[3 + i] = s;
    }
}

template <bool A, int B>
static int launch_classify(const AccumState &st, const ClsParams &P, cudaStream_t s) {
    static bool attr_done = false;
    if (!attr_done) {
        B3C_CUDA(cudaFuncSetAttribute(k_classify<A, B>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_MAX));
        attr_done = true;
    }
    k_classify<A, B><<<st.cls_grid, CLS_THREADS, st.cls_smem, s>>>(P);
    B3C_LAUNCH_CHECK();
    return B3C_OK;
}

static int get_state(void *ws, AccumState *out) {
    std::lock_guard<std::mutex> g(g_mu);
    auto it = g_states.find(ws);
    if (it == g_states.end()) {
        set_error("workspace %p has no accumulator: call b3c_accum_begin first", ws);
        return B3C_ERR_ARG;
    }
    *out = it->second;
    return B3C_OK;
}

}  // namespace b3c

using namespace b3c;

extern "C" {

int64_t b3c_accum_workspace_bytes(int64_t pair_capacity, int32_t n_seq, int32_t n_refs) {
    if (pair_capacity < 0 || n_seq <= 0 || n_refs <= 0) return B3C_ERR_ARG;
    AccumState st;
    plan(st, pair_capacity, n_seq, n_refs);
    return st.total;
}

int b3c_accum_plan(int64_t pair_capacity, int32_t n_seq, int32_t n_refs, int64_t *h_out) {
    B3C_REQUIRE(h_out != nullptr && pair_capacity >= 0 && n_seq > 0 && n_refs > 0, "bad arguments");
    AccumState st;
    plan(st, pair_capacity, n_seq, n_refs);
    h_out[0] = st.b;
    h_out[1] = st.smem_diag ? 1 : 0;
    h_out[2] = st.smem_rank;
    h_out[3] = st.cls_cap_w;
    h_out[4] = st.cls_diag_k;
    h_out[5] = radix_passes(2 * st.b);              // key sort, bits [0, 2b)
    h_out[6] = radix_digit(2 * st.b);
    h_out[7] = radix_passes(st.b);                  // composite sort, its b column bits
    h_out[8] = radix_digit(st.b);
    h_out[9] = comp_cbits(st.b);
    return B3C_OK;
}

int b3c_accum_begin(void *d_ws, int64_t ws_bytes, int64_t pair_capacity, int32_t n_seq,
                    const int32_t *d_tid2idx, int32_t n_refs, void *stream) {
    B3C_REQUIRE(d_ws && d_tid2idx, "null pointer");
    B3C_REQUIRE(n_seq > 0 && n_refs > 0 && pair_capacity >= 0, "invalid sizes N=%d refs=%d cap=%lld", n_seq, n_refs,
                (long long)pair_capacity);
    B3C_REQUIRE(pair_capacity < 0xffffffffll, "pair capacity must be below 2^32 per accumulator");
    AccumState st;
    plan(st, pair_capacity, n_seq, n_refs);
    if (ws_bytes < st.total) {
        set_error("workspace too small: %lld < %lld", (long long)ws_bytes, (long long)st.total);
        return B3C_ERR_CAPACITY;
    }
    st.d_lut = d_tid2idx;
    graph_forget(d_ws);                                  // a re-planned workspace invalidates its captured sequences
    cudaStream_t s = (cudaStream_t)stream;
    char *ws = (char *)d_ws;
    B3C_CUDA(cudaMemsetAsync(ws + st.o_ctr, 0, C_COUNT * 8, s));
    B3C_CUDA(cudaMemsetAsync(ws + st.o_diag, 0, (size_t)n_seq * 4, s));
    // rank table + on-device check that tid2idx is the dense rank map
    unsigned long long one = 1;
    B3C_CUDA(cudaMemcpyAsync(ws + st.o_ctr + C_LUT_OK * 8, &one, 8, cudaMemcpyHostToDevice, s));
    int64_t *cnt64 = (int64_t *)(ws + st.o_tmp64);
    int64_t *pref64 = cnt64 + st.rank_words + 1;
    k_rank_bits<<<(unsigned)ceil_div(st.rank_words, 256), 256, 0, s>>>(d_tid2idx, n_refs, st.rank_words,
                                                                      (unsigned long long *)(ws + st.o_bits), cnt64);
    B3C_LAUNCH_CHECK();
    int rc = scan_exclusive_i64(cnt64, pref64, st.rank_words, (int64_t *)(ws + st.o_scan_tmp), s);
    if (rc) return rc;
    const int64_t nver = n_refs > st.rank_words ? n_refs : st.rank_words;
    k_rank_verify<<<(unsigned)ceil_div(nver, 256), 256, 0, s>>>(d_tid2idx, n_refs, n_seq,
                                                               (const unsigned long long *)(ws + st.o_bits), pref64,
                                                               (uint32_t *)(ws + st.o_pref), st.rank_words,
                                                               (unsigned long long *)(ws + st.o_ctr));
    B3C_LAUNCH_CHECK();
    std::lock_guard<std::mutex> g(g_mu);
    g_states[d_ws] = st;
    return B3C_OK;
}

int b3c_accum_reset(void *d_ws, void *stream) {
    AccumState st;
    int rc = get_state(d_ws, &st);
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    char *ws = (char *)d_ws;
    // keep C_LUT_OK (the rank-table verdict of begin); clear the per-map counters and the diagonal
    B3C_CUDA(cudaMemsetAsync(ws + st.o_ctr, 0, C_LUT_OK * 8, s));
    B3C_CUDA(cudaMemsetAsync(ws + st.o_ctr + (C_LUT_OK + 1) * 8, 0, (C_COUNT - C_LUT_OK - 1) * 8, s));
    B3C_CUDA(cudaMemsetAsync(ws + st.o_diag, 0, (size_t)st.n_seq * 4, s));
    st.reduced = false;
    st.nnz_uo = st.nnz_diag = 0;
    std::lock_guard<std::mutex> g(g_mu);
    g_states[d_ws] = st;
    return B3C_OK;
}

static int accum_add(void *d_ws, const void *d_records, int64_t n_records, int32_t rec_bytes, void *stream,
                     int32_t rec_same = 0);

int b3c_accum_add_pairs(void *d_ws, const uint64_t *d_records, int64_t n_records, void *stream) {
    return accum_add(d_ws, d_records, n_records, 8, stream);
}

int b3c_accum_add_pairs_packed(void *d_ws, const void *d_bytes, int64_t n_records, int32_t bytes_per_record,
                               void *stream) {
    B3C_REQUIRE(bytes_per_record == 5 || bytes_per_record == 6 || bytes_per_record == 8,
                "bytes_per_record must be 5, 6 or 8");
    return accum_add(d_ws, d_bytes, n_records, bytes_per_record, stream);
}

int b3c_accum_add_pairs_same(void *d_ws, const void *d_bytes, int64_t n_records, int32_t bytes_per_record,
                             void *stream) {
    B3C_REQUIRE(bytes_per_record == 3 || bytes_per_record == 4, "bytes_per_record must be 3 or 4");
    return accum_add(d_ws, d_bytes, n_records, bytes_per_record, stream, 1);
}

static int accum_add(void *d_ws, const void *d_records_v, int64_t n_records, int32_t rec_bytes, void *stream,
                     int32_t rec_same) {
    const uint64_t *d_records = (const uint64_t *)d_records_v;
    AccumState st;
    int rc = get_state(d_ws, &st);
    if (rc) return rc;
    B3C_REQUIRE(n_records >= 0, "negative record count");
    if (n_records == 0) return B3C_OK;
    B3C_REQUIRE(d_records != nullptr, "null records");
    B3C_REQUIRE(((uintptr_t)d_records & 15) == 0, "records must be 16-byte aligned");
    if (rec_bytes != 8) {
        const int tb = rec_same ? 8 * rec_bytes - 1 : (8 * rec_bytes - 1) / 2;
        B3C_REQUIRE((int64_t)st.n_refs < (1ll << tb) - 1, "%d-byte records hold reference ids below %lld; the table has %d",
                    rec_bytes, (1ll << tb) - 1, st.n_refs);
    }
    B3C_REQUIRE(!st.reduced, "accumulator already reduced: call b3c_accum_begin to start a new map");
    char *ws = (char *)d_ws;
    ClsParams P;
    P.rec = d_records;
    P.n_rec = n_records;
    P.rec_bytes = rec_bytes;
    P.rec_same = rec_same;
    P.lut = st.d_lut;
    P.n_refs = st.n_refs;
    P.n_seq = st.n_seq;
    P.b = st.b;
    P.rank_words = st.rank_words;
    P.g_bits = (const unsigned long long *)(ws + st.o_bits);
    P.g_pref = (const uint32_t *)(ws + st.o_pref);
    P.diag = (uint32_t *)(ws + st.o_diag);
    P.keys = (uint64_t *)(ws + st.o_keys_a);
    P.cap = st.cap;
    P.ctr = (unsigned long long *)(ws + st.o_ctr);
    P.cap_w = st.cls_cap_w;
    P.diag_k = st.cls_diag_k;
    cudaStream_t s = (cudaStream_t)stream;
    if (st.smem_diag) {
        if (st.smem_rank == 3) return launch_classify<true, 3>(st, P, s);
        if (st.smem_rank == 2) return launch_classify<true, 2>(st, P, s);
        if (st.smem_rank == 1) return launch_classify<true, 1>(st, P, s);
        return launch_classify<true, 0>(st, P, s);
    }
    if (st.smem_rank == 3) return launch_classify<false, 3>(st, P, s);
    if (st.smem_rank == 2) return launch_classify<false, 2>(st, P, s);
    if (st.smem_rank == 1) return launch_classify<false, 1>(st, P, s);
    return launch_classify<false, 0>(st, P, s);
}

int b3c_accum_reduce(void *d_ws, int64_t *h_sizes, void *stream) {
    AccumState st;
    int rc = get_state(d_ws, &st);
    if (rc) return rc;
    B3C_REQUIRE(h_sizes != nullptr, "null h_sizes");
    cudaStream_t s = (cudaStream_t)stream;
    char *ws = (char *)d_ws;
    unsigned long long *ctr = (unsigned long long *)(ws + st.o_ctr);
    uint64_t *ka = (uint64_t *)(ws + st.o_keys_a), *kb = (uint64_t *)(ws + st.o_keys_b);
    uint64_t *uniq = (uint64_t *)(ws + st.o_uniq);
    uint32_t *pos = (uint32_t *)(ws + st.o_pos), *cnt = (uint32_t *)(ws + st.o_cnt);
    uint32_t *hist = (uint32_t *)(ws + st.o_hist);
    int64_t *heads = (int64_t *)(ws + st.o_heads), *heads_ex = heads + RS_BLOCKS + 2;
    int64_t *scan_tmp = (int64_t *)(ws + st.o_scan_tmp);
    uint32_t *diag = (uint32_t *)(ws + st.o_diag);
    int64_t *up = (int64_t *)(ws + st.o_up_ptr), *lo = (int64_t *)(ws + st.o_lo_ptr), *len = (int64_t *)(ws + st.o_len);
    int64_t *ip_f = (int64_t *)(ws + st.o_indptr_f), *ip_u = (int64_t *)(ws + st.o_indptr_u);

    rc = radix_init();
    if (rc) return rc;
    // where the two sorts leave their results is a function of the key width alone
    uint64_t *sorted = radix_where(0, 2 * st.b) ? kb : ka, *other = radix_where(0, 2 * st.b) ? ka : kb;
    const int csh = st.b + comp_cbits(st.b);             // the column j sits in bits [csh, csh + b) of a composite
    uint64_t *comp = radix_where(csh, csh + st.b) ? other : sorted;
    st.comp_in_a = (comp == ka) ? 1 : 0;
    // The whole sequence (~60 launches; every size is read from device counters) is one CUDA graph per workspace.
    rc = graph_run(s, d_ws, /*id*/ 1, nullptr, [&]() -> int {
        int where = 0, rc2;
        k_accum_guard<<<1, 1, 0, s>>>(ctr, st.cap);
        B3C_LAUNCH_CHECK();
        // 1. sort the off-diagonal keys on their 2b significant bits
        rc2 = radix_sort(ka, kb, ctr + C_NKEYS, 0, 2 * st.b, hist, s, &where);
        if (rc2) return rc2;
        // 2. run-length reduce -> unique keys + counts, composite (j, e) for the mirror half
        k_rle_count<<<RS_BLOCKS, RS_THREADS, 0, s>>>(sorted, ctr + C_NKEYS, heads);
        B3C_LAUNCH_CHECK();
        rc2 = scan_exclusive_i64(heads, heads_ex, RS_BLOCKS, scan_tmp, s);
        if (rc2) return rc2;
        k_rle_write<<<RS_BLOCKS, RS_THREADS, 0, s>>>(sorted, ctr + C_NKEYS, heads_ex, uniq, pos);
        B3C_LAUNCH_CHECK();
        k_rle_finish<<<1, 1, 0, s>>>(heads_ex, RS_BLOCKS, ctr + C_NKEYS, pos, ctr);
        B3C_LAUNCH_CHECK();
        k_rle_counts<<<kNumSMs * 8, 256, 0, s>>>(pos, ctr, cnt, st.b, uniq, sorted);   // composite overwrites the sorted keys
        B3C_LAUNCH_CHECK();
        k_diag_stats<<<kNumSMs * 2, 256, 0, s>>>(diag, st.n_seq, ctr);
        B3C_LAUNCH_CHECK();
        // 3. stable sort of the composite on the column bits only -> (j, i) order
        rc2 = radix_sort(sorted, other, ctr + C_NNZ_UO, csh, csh + st.b, hist, s, &where);
        if (rc2) return rc2;
        // 4. row pointers of both halves, row lengths, indptr of both output forms
        k_row_ptr<<<kNumSMs * 8, 256, 0, s>>>(uniq, ctr + C_NNZ_UO, st.b, st.n_seq, up);
        B3C_LAUNCH_CHECK();
        k_row_ptr<<<kNumSMs * 8, 256, 0, s>>>(comp, ctr + C_NNZ_UO, csh, st.n_seq, lo);
        B3C_LAUNCH_CHECK();
        k_row_len<<<kNumSMs * 4, 256, 0, s>>>(up, lo, diag, st.n_seq, len, ip_u /* scratch: upper lengths */);
        B3C_LAUNCH_CHECK();
        rc2 = scan_exclusive_i64(len, ip_f, st.n_seq, scan_tmp, s);
        if (rc2) return rc2;
        B3C_CUDA(cudaMemcpyAsync(len, ip_u, (size_t)st.n_seq * 8, cudaMemcpyDeviceToDevice, s));
        return scan_exclusive_i64(len, ip_u, st.n_seq, scan_tmp, s);
    });
    if (rc) return rc;

    unsigned long long h[C_COUNT];
    B3C_CUDA(cudaMemcpyAsync(h, ctr, sizeof(h), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaStreamSynchronize(s));
    if (h[C_OVERFLOW]) {
        set_error("pair capacity %lld exceeded by the off-diagonal keys", (long long)st.cap);
        return B3C_ERR_CAPACITY;
    }
    st.reduced = true;
    st.nnz_uo = (int64_t)h[C_NNZ_UO];
    st.nnz_diag = (int64_t)h[C_NNZ_DIAG];
    h_sizes[0] = st.nnz_uo + st.nnz_diag;
    h_sizes[1] = 2 * st.nnz_uo + st.nnz_diag;
    h_sizes[2] = (int64_t)h[C_ACCEPT];
    h_sizes[3] = (int64_t)h[C_EXCL];
    h_sizes[4] = (int64_t)h[C_POOR];
    h_sizes[5] = (int64_t)h[C_WEIGHT];
    std::lock_guard<std::mutex> g(g_mu);
    g_states[d_ws] = st;
    return B3C_OK;
}

int b3c_accum_emit_csr(void *d_ws, int symmetric, int64_t *d_indptr, int32_t *d_indices, uint32_t *d_counts,
                       void *stream) {
    AccumState st;
    int rc = get_state(d_ws, &st);
    if (rc) return rc;
    B3C_REQUIRE(st.reduced, "call b3c_accum_reduce before b3c_accum_emit_csr");
    B3C_REQUIRE(d_indptr != nullptr, "null indptr");
    const int64_t nnz_out = symmetric ? 2 * st.nnz_uo + st.nnz_diag : st.nnz_uo + st.nnz_diag;
    B3C_REQUIRE(nnz_out == 0 || (d_indices && d_counts), "null output arrays");
    cudaStream_t s = (cudaStream_t)stream;
    char *ws = (char *)d_ws;
    const int64_t *ip = (const int64_t *)(ws + (symmetric ? st.o_indptr_f : st.o_indptr_u));
    B3C_CUDA(cudaMemcpyAsync(d_indptr, ip, ((size_t)st.n_seq + 1) * 8, cudaMemcpyDeviceToDevice, s));
    k_emit<<<kNumSMs * 8, 256, 0, s>>>(symmetric ? 1 : 0, st.b, st.n_seq, (const unsigned long long *)(ws + st.o_ctr),
                                       (const uint64_t *)(ws + st.o_uniq), (const uint32_t *)(ws + st.o_cnt),
                                       (const uint64_t *)(ws + (st.comp_in_a ? st.o_keys_a : st.o_keys_b)),
                                       (const uint32_t *)(ws + st.o_diag), (const int64_t *)(ws + st.o_up_ptr),
                                       (const int64_t *)(ws + st.o_lo_ptr), ip, d_indices, d_counts);
    B3C_LAUNCH_CHECK();
    return B3C_OK;
}

// ---- sharded accumulation entry points (see bin3c_b200/dist.py) ---------------------------------------

int b3c_accum_offsets(void *d_ws, int64_t *h_offsets) {
    AccumState st;
    int rc = get_state(d_ws, &st);
    if (rc) return rc;
    B3C_REQUIRE(h_offsets != nullptr, "null h_offsets");
    h_offsets[0] = st.o_ctr;       // uint64[16] counters
    h_offsets[1] = st.o_diag;      // uint32[n_seq] diagonal counts
    h_offsets[2] = st.o_keys_a;    // uint64[cap] canonical keys after add_pairs
    h_offsets[3] = st.cap;
    return B3C_OK;
}

int b3c_accum_row_hist(void *d_ws, uint64_t *d_rowcnt, void *stream) {
    AccumState st;
    int rc = get_state(d_ws, &st);
    if (rc) return rc;
    B3C_REQUIRE(d_rowcnt != nullptr, "null rowcnt");
    char *ws = (char *)d_ws;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long *ctr = (unsigned long long *)(ws + st.o_ctr);
    k_accum_guard<<<1, 1, 0, s>>>(ctr, st.cap);
    B3C_LAUNCH_CHECK();
    k_row_hist<<<kNumSMs * 8, 256, 0, s>>>((const uint64_t *)(ws + st.o_keys_a), ctr + C_NKEYS, st.b,
                                           (unsigned long long *)d_rowcnt);
    B3C_LAUNCH_CHECK();
    return B3C_OK;
}

int b3c_accum_route(void *d_ws, const int32_t *d_splits, int32_t n_ranks, uint64_t *d_out, int64_t out_capacity,
                    uint64_t *d_scratch, int64_t *h_counts, void *stream) {
    AccumState st;
    int rc = get_state(d_ws, &st);
    if (rc) return rc;
    B3C_REQUIRE(d_splits && d_out && d_scratch && h_counts, "null pointer");
    B3C_REQUIRE(n_ranks >= 1 && n_ranks <= ROUTE_MAX_RANKS, "unsupported rank count %d", n_ranks);
    char *ws = (char *)d_ws;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long *ctr = (unsigned long long *)(ws + st.o_ctr);
    const uint64_t *keys = (const uint64_t *)(ws + st.o_keys_a);
    unsigned long long *cnt = (unsigned long long *)d_scratch;              // [G]
    unsigned long long *base = cnt + ROUTE_MAX_RANKS;                       // [G+1]
    unsigned long long *cursor = base + ROUTE_MAX_RANKS + 1;                // [G]
    B3C_CUDA(cudaMemsetAsync(d_scratch, 0, (3 * ROUTE_MAX_RANKS + 2) * 8, s));
    k_accum_guard<<<1, 1, 0, s>>>(ctr, st.cap);
    B3C_LAUNCH_CHECK();
    k_route_count<<<kNumSMs * 4, 256, 0, s>>>(keys, ctr + C_NKEYS, st.b, d_splits, n_ranks, cnt);
    B3C_LAUNCH_CHECK();
    k_route_bases<<<1, 32, 0, s>>>(cnt, n_ranks, base, cursor);
    B3C_LAUNCH_CHECK();
    unsigned long long h[ROUTE_MAX_RANKS + 1 + C_COUNT];
    B3C_CUDA(cudaMemcpyAsync(h, base, (n_ranks + 1) * 8, cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaMemcpyAsync(h + ROUTE_MAX_RANKS + 1, ctr, C_COUNT * 8, cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaStreamSynchronize(s));
    if (h[ROUTE_MAX_RANKS + 1 + C_OVERFLOW]) {
        set_error("pair capacity %lld exceeded by the off-diagonal keys", (long long)st.cap);
        return B3C_ERR_CAPACITY;
    }
    if ((int64_t)h[n_ranks] > out_capacity) {
        set_error("route buffer too small: %llu > %lld", h[n_ranks], (long long)out_capacity);
        return B3C_ERR_CAPACITY;
    }
    k_route_scatter<<<kNumSMs * 4, 256, 0, s>>>(keys, ctr + C_NKEYS, st.b, d_splits, n_ranks, cursor, d_out);
    B3C_LAUNCH_CHECK();
    for (int g = 0; g <= n_ranks; ++g) h_counts[g] = (int64_t)h[g];          // exclusive offsets, [G] = total
    // local pair counters ride along: accepted, ref_excluded, poor_match
    h_counts[n_ranks + 1] = (int64_t)h[ROUTE_MAX_RANKS + 1 + C_ACCEPT];
    h_counts[n_ranks + 2] = (int64_t)h[ROUTE_MAX_RANKS + 1 + C_EXCL];
    h_counts[n_ranks + 3] = (int64_t)h[ROUTE_MAX_RANKS + 1 + C_POOR];
    return B3C_OK;
}

int b3c_accum_reduce_block(void *d_ws, const uint64_t *d_keys, int64_t n_keys, int32_t row_lo, int32_t row_hi,
                           int64_t *h_sizes, void *stream) {
    AccumState st;
    int rc = get_state(d_ws, &st);
    if (rc) return rc;
    B3C_REQUIRE(h_sizes != nullptr && n_keys >= 0, "bad arguments");
    B3C_REQUIRE(0 <= row_lo && row_lo < row_hi && row_hi <= st.n_seq, "bad row block [%d,%d)", row_lo, row_hi);
    if (n_keys > st.cap) {
        set_error("received %lld directed keys, accumulator capacity is %lld", (long long)n_keys, (long long)st.cap);
        return B3C_ERR_CAPACITY;
    }
    cudaStream_t s = (cudaStream_t)stream;
    char *ws = (char *)d_ws;
    unsigned long long *ctr = (unsigned long long *)(ws + st.o_ctr);
    uint64_t *ka = (uint64_t *)(ws + st.o_keys_a), *kb = (uint64_t *)(ws + st.o_keys_b);
    uint64_t *uniq = (uint64_t *)(ws + st.o_uniq);
    uint32_t *pos = (uint32_t *)(ws + st.o_pos), *cnt = (uint32_t *)(ws + st.o_cnt);
    uint32_t *hist = (uint32_t *)(ws + st.o_hist);
    int64_t *heads = (int64_t *)(ws + st.o_heads), *heads_ex = heads + RS_BLOCKS + 2;
    int64_t *scan_tmp = (int64_t *)(ws + st.o_scan_tmp);
    uint32_t *diag = (uint32_t *)(ws + st.o_diag);
    int64_t *ptr = (int64_t *)(ws + st.o_up_ptr), *len = (int64_t *)(ws + st.o_len);
    int64_t *ip = (int64_t *)(ws + st.o_indptr_f);
    const int32_t n_local = row_hi - row_lo;

    if (n_keys) B3C_CUDA(cudaMemcpyAsync(ka, d_keys, (size_t)n_keys * 8, cudaMemcpyDeviceToDevice, s));
    const unsigned long long nk = (unsigned long long)n_keys;
    B3C_CUDA(cudaMemcpyAsync(ctr + C_NKEYS, &nk, 8, cudaMemcpyHostToDevice, s));
    B3C_CUDA(cudaMemsetAsync(ctr + C_NNZ_UO, 0, 3 * 8, s));       // nnz_uo, nnz_diag, weight
    rc = radix_init();
    if (rc) return rc;
    int where = 0;
    rc = radix_sort(ka, kb, ctr + C_NKEYS, 0, 2 * st.b, hist, s, &where);
    if (rc) return rc;
    uint64_t *sorted = where ? kb : ka;
    k_rle_count<<<RS_BLOCKS, RS_THREADS, 0, s>>>(sorted, ctr + C_NKEYS, heads);
    B3C_LAUNCH_CHECK();
    rc = scan_exclusive_i64(heads, heads_ex, RS_BLOCKS, scan_tmp, s);
    if (rc) return rc;
    k_rle_write<<<RS_BLOCKS, RS_THREADS, 0, s>>>(sorted, ctr + C_NKEYS, heads_ex, uniq, pos);
    B3C_LAUNCH_CHECK();
    k_rle_finish<<<1, 1, 0, s>>>(heads_ex, RS_BLOCKS, ctr + C_NKEYS, pos, ctr);
    B3C_LAUNCH_CHECK();
    k_rle_counts<<<kNumSMs * 8, 256, 0, s>>>(pos, ctr, cnt, st.b, uniq, sorted);
    B3C_LAUNCH_CHECK();
    k_row_ptr<<<kNumSMs * 8, 256, 0, s>>>(uniq, ctr + C_NNZ_UO, st.b, st.n_seq, ptr);
    B3C_LAUNCH_CHECK();
    k_block_row_len<<<(unsigned)ceil_div(n_local, 256), 256, 0, s>>>(ptr, diag, row_lo, n_local, len);
    B3C_LAUNCH_CHECK();
    rc = scan_exclusive_i64(len, ip, n_local, scan_tmp, s);
    if (rc) return rc;
    int64_t nnz_local = 0;
    B3C_CUDA(cudaMemcpyAsync(&nnz_local, ip + n_local, 8, cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaStreamSynchronize(s));
    st.reduced = true;
    st.nnz_uo = nnz_local;
    h_sizes[0] = nnz_local;
    std::lock_guard<std::mutex> g(g_mu);
    g_states[d_ws] = st;
    return B3C_OK;
}

int b3c_accum_emit_block(void *d_ws, int32_t row_lo, int32_t row_hi, int64_t *d_indptr, int32_t *d_indices,
                         uint32_t *d_counts, void *stream) {
    AccumState st;
    int rc = get_state(d_ws, &st);
    if (rc) return rc;
    B3C_REQUIRE(st.reduced, "call b3c_accum_reduce_block first");
    B3C_REQUIRE(d_indptr != nullptr && 0 <= row_lo && row_lo < row_hi && row_hi <= st.n_seq, "bad arguments");
    cudaStream_t s = (cudaStream_t)stream;
    char *ws = (char *)d_ws;
    const int32_t n_local = row_hi - row_lo;
    const int64_t *ip = (const int64_t *)(ws + st.o_indptr_f);
    B3C_CUDA(cudaMemcpyAsync(d_indptr, ip, ((size_t)n_local + 1) * 8, cudaMemcpyDeviceToDevice, s));
    const int64_t blocks = (int64_t)kNumSMs * 16;          // grid-stride over the block's entries, then its rows
    k_emit_block<<<(unsigned)blocks, 256, 0, s>>>(st.b, row_lo, n_local, (const uint64_t *)(ws + st.o_uniq),
                                                  (const uint32_t *)(ws + st.o_cnt), (const uint32_t *)(ws + st.o_diag),
                                                  (const int64_t *)(ws + st.o_up_ptr), ip, d_indices, d_counts);
    B3C_LAUNCH_CHECK();
    return B3C_OK;
}

// ---- peer exchange arena entry points -----------------------------------------------------------------

static int peers_of(void *const *h_arena, int32_t rank, int32_t n_ranks, Peers *P) {
    B3C_REQUIRE(h_arena != nullptr && n_ranks >= 1 && n_ranks <= XA_MAX_RANKS && rank >= 0 && rank < n_ranks,
                "bad rank %d of %d (at most %d)", rank, n_ranks, XA_MAX_RANKS);
    for (int g = 0; g < XA_MAX_RANKS; ++g) P->a[g] = nullptr;
    for (int g = 0; g < n_ranks; ++g) {
        B3C_REQUIRE(h_arena[g] != nullptr, "null arena of rank %d", g);
        P->a[g] = (char *)h_arena[g];
    }
    return B3C_OK;
}

int64_t b3c_xa_bytes(int32_t n_seq, int64_t key_capacity) {
    if (n_seq <= 0 || key_capacity < 0) return B3C_ERR_ARG;
    return xa_layout(n_seq, key_capacity).total;
}

int b3c_xa_offsets(int32_t n_seq, int64_t key_capacity, int64_t *h_offsets) {
    B3C_REQUIRE(n_seq > 0 && key_capacity >= 0 && h_offsets, "bad arguments");
    const XaLayout X = xa_layout(n_seq, key_capacity);
    h_offsets[0] = X.o_mask;
    h_offsets[1] = X.o_x;
    h_offsets[2] = X.o_keys;
    h_offsets[3] = X.o_diag;
    return B3C_OK;
}

int b3c_peer_barrier(void *const *h_arena, int32_t rank, int32_t n_ranks, int32_t n_seq, int64_t key_capacity,
                     uint64_t epoch, void *stream) {
    Peers P;
    int rc = peers_of(h_arena, rank, n_ranks, &P);
    if (rc) return rc;
    const XaLayout X = xa_layout(n_seq, key_capacity);
    k_peer_barrier<<<1, 32, 0, (cudaStream_t)stream>>>(P, rank, n_ranks, epoch, X.o_flag, X.o_ctl,
                                                       g_peer_timeout_cycles.load());
    B3C_LAUNCH_CHECK();
    return B3C_OK;
}

int b3c_peer_put(void *const *h_arena, int32_t n_ranks, int64_t offset, const void *d_src, int64_t bytes, void *stream) {
    Peers P;
    int rc = peers_of(h_arena, 0, n_ranks, &P);
    if (rc) return rc;
    B3C_REQUIRE(offset >= 0 && bytes >= 0 && (bytes == 0 || d_src), "bad arguments");
    if (bytes == 0) return B3C_OK;
    int64_t blocks = ceil_div(bytes, 16 * 256);
    if (blocks > kNumSMs * 4) blocks = kNumSMs * 4;
    k_peer_put<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(P, n_ranks, offset, (const unsigned char *)d_src, bytes);
    B3C_LAUNCH_CHECK();
    return B3C_OK;
}

int b3c_peer_allreduce_f64(void *const *h_arena, int32_t rank, int32_t n_ranks, int32_t n_seq, int64_t key_capacity,
                           uint64_t epoch, int32_t op, double *d_val, int32_t count, void *stream) {
    Peers P;
    int rc = peers_of(h_arena, rank, n_ranks, &P);
    if (rc) return rc;
    B3C_REQUIRE(d_val && count >= 1 && count <= XA_SCAL && (op == 0 || op == 1), "bad arguments");
    const XaLayout X = xa_layout(n_seq, key_capacity);
    k_peer_allreduce<<<1, 64, 0, (cudaStream_t)stream>>>(P, rank, n_ranks, epoch, op, d_val, count, X.o_flag, X.o_ctl,
                                                         X.o_scal, g_peer_timeout_cycles.load());
    B3C_LAUNCH_CHECK();
    return B3C_OK;
}

int b3c_shard_publish(void *d_ws, void *const *h_arena, int32_t rank, int32_t n_ranks, void *stream) {
    AccumState st;
    int rc = get_state(d_ws, &st);
    if (rc) return rc;
    Peers P;
    rc = peers_of(h_arena, rank, n_ranks, &P);
    if (rc) return rc;
    const XaLayout X = xa_layout(st.n_seq, st.cap);
    cudaStream_t s = (cudaStream_t)stream;
    char *ws = (char *)d_ws;
    unsigned long long *ctr = (unsigned long long *)(ws + st.o_ctr);
    char *mine = P.a[rank];
    k_accum_guard<<<1, 1, 0, s>>>(ctr, st.cap);
    B3C_LAUNCH_CHECK();
    // receive cursor, overflow word and time-out word of this rank (nobody scatters to it before the next barrier;
    // the time-out word is only ever set by this rank's own kernels, so a reported time-out does not outlive a run)
    B3C_CUDA(cudaMemsetAsync(mine + X.o_ctl, 0, 24, s));
    // chunk weights of the local keys, accumulated in this rank's own slot, then copied to every other arena
    unsigned long long *cw = (unsigned long long *)(mine + X.o_cw) + (int64_t)rank * X.n_chunks;
    B3C_CUDA(cudaMemsetAsync(cw, 0, (size_t)X.n_chunks * 8, s));
    const int smem = X.n_chunks <= XA_MAX_CHUNKS ? X.n_chunks * 4 : 0;
    static bool attr_done = false;
    if (!attr_done) {
        B3C_CUDA(cudaFuncSetAttribute(k_chunk_weights, cudaFuncAttributeMaxDynamicSharedMemorySize, XA_MAX_CHUNKS * 4));
        attr_done = true;
    }
    k_chunk_weights<<<kNumSMs * 4, 256, smem, s>>>((const uint64_t *)(ws + st.o_keys_a), ctr + C_NKEYS, st.b, X.n_chunks, cw);
    B3C_LAUNCH_CHECK();
    if (n_ranks > 1) {
        Peers others = P;
        k_peer_put<<<8, 256, 0, s>>>(others, n_ranks, X.o_cw + (int64_t)rank * X.n_chunks * 8, (const unsigned char *)cw,
                                     (int64_t)X.n_chunks * 8);
        B3C_LAUNCH_CHECK();
    }
    k_publish_counters<<<1, 32, 0, s>>>(P, rank, n_ranks, ctr, X.o_cnt3);
    B3C_LAUNCH_CHECK();
    // the local diagonal histogram, where the owners of the rows can read it
    B3C_CUDA(cudaMemcpyAsync(mine + X.o_diag, ws + st.o_diag, (size_t)st.n_seq * 4, cudaMemcpyDeviceToDevice, s));
    return B3C_OK;
}

int b3c_shard_scatter(void *d_ws, void *const *h_arena, int32_t rank, int32_t n_ranks, int32_t *d_splits, void *stream) {
    AccumState st;
    int rc = get_state(d_ws, &st);
    if (rc) return rc;
    Peers P;
    rc = peers_of(h_arena, rank, n_ranks, &P);
    if (rc) return rc;
    B3C_REQUIRE(d_splits != nullptr, "null splits");
    const XaLayout X = xa_layout(st.n_seq, st.cap);
    if (X.n_chunks > XA_MAX_CHUNKS) {
        set_error("sharded accumulation supports at most %d row chunks (%d contigs)", XA_MAX_CHUNKS, XA_MAX_CHUNKS * XA_CHUNK);
        return B3C_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    char *ws = (char *)d_ws;
    unsigned long long *ctr = (unsigned long long *)(ws + st.o_ctr);
    k_shard_splits<<<1, 1024, 0, s>>>(P, rank, n_ranks, st.n_seq, X.n_chunks, X.o_cw, d_splits);
    B3C_LAUNCH_CHECK();
    k_route_peer<<<kNumSMs * 4, RT_THREADS, 0, s>>>((const uint64_t *)(ws + st.o_keys_a), ctr + C_NKEYS, st.b, d_splits, P,
                                                    n_ranks, X.o_ctl, X.o_keys, st.cap);
    B3C_LAUNCH_CHECK();
    return B3C_OK;
}

int b3c_shard_reduce_block(void *d_ws, void *const *h_arena, int32_t rank, int32_t n_ranks, const int32_t *d_splits,
                           int64_t *h_sizes, void *stream) {
    AccumState st;
    int rc = get_state(d_ws, &st);
    if (rc) return rc;
    Peers P;
    rc = peers_of(h_arena, rank, n_ranks, &P);
    if (rc) return rc;
    B3C_REQUIRE(d_splits && h_sizes, "null pointer");
    const XaLayout X = xa_layout(st.n_seq, st.cap);
    cudaStream_t s = (cudaStream_t)stream;
    char *ws = (char *)d_ws;
    unsigned long long *ctr = (unsigned long long *)(ws + st.o_ctr);
    uint64_t *ka = (uint64_t *)(P.a[rank] + X.o_keys), *kb = (uint64_t *)(ws + st.o_keys_b);
    uint64_t *uniq = (uint64_t *)(ws + st.o_uniq);
    uint32_t *pos = (uint32_t *)(ws + st.o_pos), *cnt = (uint32_t *)(ws + st.o_cnt);
    uint32_t *hist = (uint32_t *)(ws + st.o_hist);
    int64_t *heads = (int64_t *)(ws + st.o_heads), *heads_ex = heads + RS_BLOCKS + 2;
    int64_t *scan_tmp = (int64_t *)(ws + st.o_scan_tmp);
    uint32_t *diag = (uint32_t *)(ws + st.o_diag);
    int64_t *ptr = (int64_t *)(ws + st.o_up_ptr), *len = (int64_t *)(ws + st.o_len);
    int64_t *ip = (int64_t *)(ws + st.o_indptr_f);
    unsigned long long *d_out = (unsigned long long *)(ws + st.o_tmp64);      // [6] scratch (the rank table is final)

    // the splits decide the row block: they are needed on the host to size the launches below
    int32_t h_splits[XA_MAX_RANKS + 1];
    B3C_CUDA(cudaMemcpyAsync(h_splits, d_splits, (size_t)(n_ranks + 1) * 4, cudaMemcpyDeviceToHost, s));
    rc = radix_init();
    if (rc) return rc;
    uint64_t *sorted = radix_where(0, 2 * st.b) ? kb : ka;
    // collect + sort + run-length reduce + row pointers: one CUDA graph per (workspace, arena)
    rc = graph_run(s, d_ws, /*id*/ 2, P.a[rank], [&]() -> int {
        int where = 0, rc2;
        k_shard_collect<<<1, 32, 0, s>>>(P, rank, n_ranks, X.o_ctl, X.o_cnt3, st.cap, ctr, d_out);
        B3C_LAUNCH_CHECK();
        rc2 = radix_sort(ka, kb, ctr + C_NKEYS, 0, 2 * st.b, hist, s, &where);
        if (rc2) return rc2;
        k_rle_count<<<RS_BLOCKS, RS_THREADS, 0, s>>>(sorted, ctr + C_NKEYS, heads);
        B3C_LAUNCH_CHECK();
        rc2 = scan_exclusive_i64(heads, heads_ex, RS_BLOCKS, scan_tmp, s);
        if (rc2) return rc2;
        k_rle_write<<<RS_BLOCKS, RS_THREADS, 0, s>>>(sorted, ctr + C_NKEYS, heads_ex, uniq, pos);
        B3C_LAUNCH_CHECK();
        k_rle_finish<<<1, 1, 0, s>>>(heads_ex, RS_BLOCKS, ctr + C_NKEYS, pos, ctr);
        B3C_LAUNCH_CHECK();
        k_rle_counts<<<kNumSMs * 8, 256, 0, s>>>(pos, ctr, cnt, st.b, uniq, sorted);
        B3C_LAUNCH_CHECK();
        k_row_ptr<<<kNumSMs * 8, 256, 0, s>>>(uniq, ctr + C_NNZ_UO, st.b, st.n_seq, ptr);
        B3C_LAUNCH_CHECK();
        return B3C_OK;
    });
    if (rc) return rc;
    B3C_CUDA(cudaStreamSynchronize(s));                       // h_splits
    const int32_t row_lo = h_splits[rank], row_hi = h_splits[rank + 1];
    const int32_t n_local = row_hi - row_lo;
    int64_t nnz_local = 0;
    unsigned long long h_out[6] = {0, 0, 0, 0, 0, 0};
    if (n_local > 0) {
        k_diag_gather<<<(unsigned)ceil_div(n_local, 256), 256, 0, s>>>(P, n_ranks, row_lo, row_hi, X.o_diag, diag);
        B3C_LAUNCH_CHECK();
        k_block_row_len<<<(unsigned)ceil_div(n_local, 256), 256, 0, s>>>(ptr, diag, row_lo, n_local, len);
        B3C_LAUNCH_CHECK();
        rc = scan_exclusive_i64(len, ip, n_local, scan_tmp, s);
        if (rc) return rc;
        B3C_CUDA(cudaMemcpyAsync(&nnz_local, ip + n_local, 8, cudaMemcpyDeviceToHost, s));
    }
    B3C_CUDA(cudaMemcpyAsync(h_out, d_out, sizeof(h_out), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaStreamSynchronize(s));
    if (h_out[2]) {
        set_error("sharded accumulation: a rank did not reach a barrier within the time-out");
        return B3C_ERR_CUDA;
    }
    if (h_out[1]) {
        set_error("received %llu directed keys, accumulator capacity is %lld", h_out[0], (long long)st.cap);
        return B3C_ERR_CAPACITY;
    }
    st.reduced = true;
    st.nnz_uo = nnz_local;
    h_sizes[0] = nnz_local;
    h_sizes[1] = row_lo;
    h_sizes[2] = row_hi;
    h_sizes[3] = (int64_t)h_out[3];
    h_sizes[4] = (int64_t)h_out[4];
    h_sizes[5] = (int64_t)h_out[5];
    h_sizes[6] = (int64_t)h_out[0];
    for (int g = 0; g <= n_ranks; ++g) h_sizes[8 + g] = h_splits[g];
    std::lock_guard<std::mutex> g(g_mu);
    g_states[d_ws] = st;
    return B3C_OK;
}

}  // extern "C"
