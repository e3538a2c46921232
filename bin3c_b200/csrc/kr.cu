// Knight-Ruiz balancing (sparse_utils.py:90-224) as fp64 sparse matrix-vector products + fused
// vector phases.
//
// One persistent cooperative kernel runs the whole Newton/CG iteration with device-side
// control flow: every CTA reads the same loop scalars, derived from the same per-chunk partial
// sums in the same order, so all CTAs take identical branches and the host is not involved until
// the scale vector is final.  The same phase functions are exposed one-by-one (b3c_krp_*) for
// the multi-GPU row-block driver, which puts NCCL collectives between them.
//
// SpMV operand.  A scattered fp64 gather through L1 costs one L1 wavefront per distinct 128-byte
// line (32 per warp load when the contig order is shuffled), which caps a CSR SpMV at ~1/3 of HBM
// speed on this part.  So u is gathered from SHARED memory: the columns are cut into S slabs of
// W <= 28672 entries (224 KB of fp64) and the matrix is re-laid once per balancing run as a
// slab-major STREAM: all entries of slab 0 row by row, then slab 1, ...  An entry is its fp64 value
// plus a 16-bit slab-local column: 10 B per non-zero instead of CSR's 12, and no row pointers are
// read by the SpMV at all.  Every (row, slab) segment is padded with zero entries to whole 8-entry
// PIECES, so a segment can only start at the first entry of a piece: one start flag per piece.
// The stream is cut into CHUNKS of 512 entries (two pieces per lane, stored piece-major so that a
// piece is one coalesced 64-byte-per-lane load).  A CTA -- one per SM -- owns a contiguous range
// of chunks inside ONE slab, brings that slab of u into shared memory with TMA bulk copies
// (cp.async.bulk + mbarrier), and each of its 16 warps streams its own contiguous run of chunks
// with 256-bit loads issued three pieces ahead (register ring), with no block-wide synchronisation
// inside the run.  A piece is added up as a fixed tree; a lane's pieces extend or close its open
// segment; at the end of a chunk the 32 lane runs are stitched by one segmented scan (flag counts
// from two ballots, sums by 5 shuffle steps), the warp's runs by one warp per CTA, and a segment
// that crosses a CTA's range is finished by the vector phase that consumes it, from one boundary
// record per CTA -- so the cost per entry does not depend on the row lengths (heavy-tailed contig
// rows, empty rows) and nothing is accumulated with atomics.  Matrices wider than SLAB_S_MAX slabs
// use the same stream with 32-bit columns and gather u through L1/L2 ("gather form"), unless their
// (row, slab) cells hold SLAB_DENSE_CELL entries or more on average.
//
// Vector phases.  One CTA per 1024-row chunk, two rows per thread, always the same rows in the same
// thread; every phase issues all of its L2 loads first, then computes and stores.  Four grid
// barriers per CG step (dir | SpMV | w | step); a barrier is one word: red.release to arrive (the
// release fence costs ~0.9 us: it drains the CTA's stores), ld.acquire to poll.
//
// Reductions (dot products, min, max) use fixed 1024-row chunks with a fixed tree inside the
// chunk and an in-order sum over chunks: the value does not depend on the grid size or on how
// rows are split over GPUs (row blocks are chunk aligned).
#include <cooperative_groups.h>
#include <math.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace b3c {

constexpr int KR_THREADS = 512;
constexpr int KR_WARPS = KR_THREADS / 32;
constexpr int SPMV_EPP = 8;                          // entries per lane per piece (one 64-byte load of values)
constexpr int SPMV_CHUNK = 32 * SPMV_EPP * 2;        // 512 entries per warp step: two pieces, 16 consecutive per lane
constexpr int SPMV_TILE = 2048;                      // every slab is padded to a multiple of this many entries
constexpr int CHUNK = 1024;                          // rows per reduction chunk
constexpr int CHUNK_RPT = CHUNK / KR_THREADS;
constexpr int RED_MAX = 8;                           // values reduced together by one block reduction
constexpr int SLAB_W_MAX = 28672;                    // fp64 entries of u held in shared memory (15-bit columns)
constexpr int SLAB_S_MAX = 16;                       // more slabs than this: gather form (default; B3C_OPT_KR_MAX_SLABS)
constexpr int SLAB_S_CAP = 48;                       // the most slabs the tables are sized for
constexpr int SLAB_DENSE_CELL_PACKED = 4;            // the same for the packed count stream (4 B per entry instead of 10)
constexpr int SLAB_DENSE_CELL = 6;                   // mean entries per (row, slab) cell from which slabs beyond SLAB_S_MAX pay
constexpr int KR_MAX_RANKS = 8;                      // GPUs of one node in peer mode
constexpr int BIG_CAP = 4096;                        // side list of off-diagonal counts above 65535 (packed count stream)
static_assert(KR_WARPS <= 32 && SLAB_W_MAX <= 65536, "warp records are stitched by one warp; 16-bit columns");

// partial arrays, each n_chunks long
enum { PA = 0, PB, PC, PMIN, PNEGMAX, PG1, PG2, P_COUNT };

struct KRScalars {
    double tol, delta, Delta, rt, stop_tol;
    double rho_km1, rho_km2, rout, rold, eta, inner_tol, alpha, beta, gamma;
    long long n_iter, max_iter, k, outer, n_spmv, zero_diag;
    long long ovf16;           // the count pass met more than BIG_CAP off-diagonal counts above 65535: no packed stream
    long long n_big;           // off-diagonal counts above 65535 met by the count pass (their high parts go to a side list)
    int status, ymode, ysel, state;
};

// per-phase cycle counters of CTA 0 (work = its own phase time, sync = its wait at the grid barrier)
enum { T_INIT = 0, T_SPMV, T_FIX, T_RESID, T_DIR, T_W, T_STEP, T_UPDATE, T_SCALAR, T_COUNT };
struct KRTimers {
    long long work[T_COUNT], sync[T_COUNT], total;
};

// what each warp leaves for the stitching warp after its run of chunks
struct WarpRecs {
    double head[KR_WARPS];     // sum of the entries before the run's first flag (all of them if it has none)
    double tail[KR_WARPS];     // sum of the segment still open at the end of the run
    int seen[KR_WARPS];        // the run contains a segment start
    int first[KR_WARPS];       // ordinal of the first segment that starts inside the run
    int last[KR_WARPS];        // ordinal of the last one
};

// dynamic shared memory carve (bytes)
constexpr int SM_RED = 0;
constexpr int SM_REC = SM_RED + KR_WARPS * RED_MAX * 8;
constexpr int SM_CTL = SM_REC + 2 * (int)sizeof(WarpRecs);
constexpr int SM_STATE = SM_CTL + ((int)sizeof(KRScalars) + 15) / 16 * 16;
constexpr int SM_TIM = SM_STATE + 32;           // SpmvState (16 B) + the CTA's SpMV cycle counter, then the phase timers
constexpr int SM_SLAB = SM_TIM + 2 * 9 * 8;     // work[T_COUNT], sync[T_COUNT]: accumulated in shared memory, written out once
constexpr int SM_MBAR = (SM_SLAB + (SLAB_S_CAP + 2) * 4 + 7) / 8 * 8;
constexpr int SM_U = (SM_MBAR + 8 + 127) / 128 * 128;
constexpr int SM_BYTES_GATHER = SM_U;
constexpr int SM_BYTES_SLAB = SM_U + SLAB_W_MAX * 8;
static_assert(SM_REC % 8 == 0 && SM_CTL % 8 == 0 && SM_STATE % 8 == 0 && SM_TIM % 8 == 0 && SM_MBAR % 8 == 0, "shared memory carve alignment");
static_assert(SM_BYTES_SLAB <= 232448, "exceeds the 227 KB of shared memory a CTA can opt into");

struct KRArgs {
    // local row block [row_lo, row_hi) of an n x n matrix; indptr is local (0-based), columns global
    int32_t n, row_lo, row_hi;
    int64_t nnz;
    const int64_t *indptr;
    const int32_t *indices;
    const double *data;
    // counts form: data == nullptr, the value of an entry is count / (s_i * s_j) computed on the fly
    const uint32_t *cnt32;
    const int32_t *sites;
    // counts form: the stream holds the raw uint32 counts (6 B per entry with its 16-bit column instead of 10) and the
    // site normalisation is factored out of the sum, (A u)_i = (1/s_i) sum_j c_ij (u_j / s_j): the SpMV multiplies the
    // SCALED operand us = u / s (xs = x / s for a residual), rows_q applies 1/s_i.  Same sums as the reference's
    // sum_j (c_ij / (s_i s_j)) u_j up to rounding of the factors (x moves ~1e-15, far inside the 1e-9 bar).
    int32_t cnt_stream;        // 1: sval is uint32[nnzv]; 2 (slab form): sval is uint32[nnzv] of PACKED entries, the 16-bit
                               // count in the high half and the 16-bit slab-local column in the low half -- 4 B per entry,
                               // one 32-byte load per lane and piece.  The high part of a DIAGONAL count above 65535 goes
                               // into dfix (a term coefficient * operand_i added by rows_q); the high part of an
                               // OFF-DIAGONAL count above 65535 goes into a short side list sorted by (row, column) --
                               // rows_q adds hi * operand_j for the rows the list names (sign bit of dfix set) -- and the
                               // stream falls back to form 1 only if the count pass meets more than BIG_CAP of them
    int32_t *cstart;           // [nv] offset of a cell's first entry inside its CSR row (k_cell_bounds -> k_stream_fill)
    int32_t n_big;             // entries of the side list
    long long *big_e;          // [BIG_CAP] CSR positions collected by the count pass, then sorted
    int32_t *big_row, *big_col;    // [n_big] global row and column
    double *big_hi;            // [n_big] (double)(count & 0xffff0000)
    const double *inv_s;       // [n] 1 / s_j (zero site counts taken as one, Q6)
    double *us, *xs;           // scaled operands (length n; xs lives beside x, in the exchange buffer in peer mode)
    // the stream
    int32_t slab;              // 1: 16-bit columns, u gathered from shared memory; 0: 32-bit columns, gather form
    int32_t S, W, npad;        // slabs (1 in gather form), slab width, local rows padded to CHUNK
    int64_t nv;                // S * npad (row, slab) cells
    int64_t nnzv;              // entries incl. slab padding (multiple of SPMV_TILE)
    int64_t n_sch;             // stream chunks = nnzv / SPMV_CHUNK
    int32_t n_seg;             // non-empty cells = segments
    const double *sval;
    const void *scol;          // uint16[nnzv] or uint32[nnzv]
    const uint16_t *sflag;     // [n_sch * 32] start flags of each lane's 16 entries
    const int32_t *chunk_seg0; // [n_sch] ordinal of the first segment starting at or after the chunk
    const int32_t *seg_of;     // [nv] ordinal of cell (s * npad + r), -1 if empty
    const int32_t *seg_row;    // [n_seg] cell of a segment
    const int32_t *slab_c0;    // [S+1] first chunk of each slab
    double *qs;                // [n_seg] segment sums
    // one boundary record per SpMV CTA
    int32_t n_bnd;
    double *bnd_head, *bnd_tail;
    int32_t *bnd_flag, *bnd_ord, *bnd_lr;
    // build scratch
    int64_t *cnt, *vp, *ord, *scan_tmp;
    double *dfix;
    // vectors (global row indexing, length n, each 256-byte aligned)
    double *x, *v, *rk, *y0, *y1, *p, *Z, *w, *u;
    // partials [P_COUNT][n_chunks]
    double *part;
    int32_t n_chunks;
    KRScalars *ctl;
    KRTimers *timers;
    // peer mode (one persistent kernel per GPU of a node, exchange buffers mapped over NVLink): u and the
    // partials live in the exchange buffer of every rank and are written into all of them directly
    int32_t n_rank, rank;                       // n_rank <= 1: single GPU / host-driven phases
    double *xx[KR_MAX_RANKS];                   // x of every rank (own included): A.x is xx[rank]
    double *xz[KR_MAX_RANKS];                   // Z of every rank: A.Z is xz[rank]
    double *xxs[KR_MAX_RANKS];                  // x / s of every rank (counts form): A.xs is xxs[rank]
    double *xpart[KR_MAX_RANKS];                // partials of every rank
    unsigned long long *xll[KR_MAX_RANKS];      // flagged partial words (+ arrival counter) of every rank: A.ll is xll[rank]
    unsigned long long *xflag[KR_MAX_RANKS];    // barrier flags of every rank: xflag[g][r] = epoch rank r has reached
    unsigned long long *epoch;                  // this rank's epoch counter (persists across runs)
    unsigned *bar_count, *bar_gen;              // grid barrier of the persistent kernel (zeroed per run)
    int32_t opts;                               // KR_OPT_* bits (b3c_set_option)
    long long peer_timeout;                     // cycles a cross-GPU wait may last (g_peer_timeout_cycles)
    double *xout;                               // where the persistent kernel leaves the final x (all n entries)
    long long *cta_spmv;                        // [n_bnd] cycles every CTA spent inside its SpMV phases
    unsigned long long *ll;                     // [P_COUNT][n_chunks][2] flagged words: partials exchanged without a barrier
};
enum { KR_OPT_BANK_ORDER = 1, KR_OPT_SLAB_ALIGN = 2, KR_OPT_FAST_BARRIER = 4, KR_OPT_LL_PARTIALS = 8, KR_OPT_PEER_LL_W = 16,
       KR_OPT_L2_PREFETCH = 32, KR_OPT_L2_PREFETCH_FAR = 64, KR_OPT_PIECE_SPREAD = 128 };

// What crosses the NVLink in peer mode: the owner of row r writes x[r] (once per Newton update) and Z[r] (once per CG
// step) straight into every rank's copy, and its chunk partials likewise.  Every rank then derives p and u = x * p for
// ALL columns itself (phase_dir_all), so a CG step needs two cross-GPU hand-overs (after `w`: the p.w partials; after
// `step`: Z and the remaining partials) instead of the three it took when u was what the ranks exchanged.
__device__ __forceinline__ void put_x(const KRArgs &A, int64_t r, double v) {
    A.x[r] = v;
    for (int g = 0; g < A.n_rank; ++g)
        if (g != A.rank) A.xx[g][r] = v;
    if (A.cnt_stream) {                                // the residual SpMV multiplies x / s
        const double vs = __dmul_rn(v, __ldg(A.inv_s + r));
        A.xs[r] = vs;
        for (int g = 0; g < A.n_rank; ++g)
            if (g != A.rank) A.xxs[g][r] = vs;
    }
}
__device__ __forceinline__ void put_z(const KRArgs &A, int64_t r, double v) {
    A.Z[r] = v;
    for (int g = 0; g < A.n_rank; ++g)
        if (g != A.rank) A.xz[g][r] = v;
}
// host-driven form (b3c_krp_*): the driver all-reduces u between the phases
__device__ __forceinline__ void put_u(const KRArgs &A, int64_t r, double v) { A.u[r] = v; }
// `loc`: the chunk belongs to this rank.  Without peers the other chunks get the identity (the host
// driver all-reduces the arrays); with peers their owners write them.
// `ll_epoch` != 0 (single GPU, KR_OPT_LL_PARTIALS): the partial is published as two flagged 8-byte words -- (low
// half, epoch) and (high half, epoch) -- that a reader polls until both carry the epoch it expects.  An aligned
// 8-byte store is single-copy atomic, so the value needs no fence and the phase no grid barrier: the phases that
// only produce partials (resid, w, step) hand over through these words alone, because every vector they touch is
// private to the thread that owns the row.
__device__ __forceinline__ void put_part(const KRArgs &A, int which, int c, double v, bool loc, double identity,
                                         unsigned ll_epoch = 0) {
    const int64_t i = (int64_t)which * A.n_chunks + c;
    if (ll_epoch) {
        const unsigned long long b = (unsigned long long)__double_as_longlong(v), e = (unsigned long long)ll_epoch << 32;
        if (A.n_rank <= 1) {
            asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(A.ll + 2 * i), "l"((b & 0xffffffffull) | e),
                         "l"((b >> 32) | e)
                         : "memory");
        } else if (loc) {                              // peer mode: the owner writes the words of every rank
            for (int g = 0; g < A.n_rank; ++g)
                asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(A.xll[g] + 2 * i),
                             "l"((b & 0xffffffffull) | e), "l"((b >> 32) | e)
                             : "memory");
        }
    } else if (A.n_rank <= 1) {
        A.part[i] = loc ? v : identity;
    } else if (loc) {
        for (int g = 0; g < A.n_rank; ++g) A.xpart[g][i] = v;
    }
}
// The flagged words carry the data; WAITING for them is done on one counter polled by one thread per CTA (thousands
// of threads polling the words themselves queue up in front of the writers at the L2 slices that hold them).  The
// counter is only a hint -- its relaxed add is not ordered after the words -- so readers still check the epochs.
__device__ __forceinline__ unsigned *ll_counter_of(const KRArgs &A, unsigned long long *ll) {
    return (unsigned *)(ll + 2 * (int64_t)P_COUNT * A.n_chunks);
}
__device__ __forceinline__ unsigned *ll_counter(const KRArgs &A) { return ll_counter_of(A, A.ll); }
// one arrival per chunk and hand-over, at every rank that will read the chunk's words
__device__ __forceinline__ void ll_arrive(const KRArgs &A) {
    if (A.n_rank <= 1) {
        asm volatile("red.relaxed.gpu.global.add.u32 [%0], 1;" ::"l"(ll_counter(A)) : "memory");
    } else {
        for (int g = 0; g < A.n_rank; ++g)
            asm volatile("red.relaxed.sys.global.add.u32 [%0], 1;" ::"l"(ll_counter_of(A, A.xll[g])) : "memory");
    }
}
// A peer that never writes (it failed) must not hang the node: both waits give up after the peer time-out and poison
// the result with NaN, as the flag barrier does.
__device__ __forceinline__ void ll_wait(const KRArgs &A, unsigned target) {
    if (threadIdx.x == 0) {
        unsigned seen;
        const long long t0 = clock64();
        do {
            asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(ll_counter(A)) : "memory");
            if ((int)(seen - target) < 0 && A.n_rank > 1 && clock64() - t0 > A.peer_timeout) {
                A.timers->sync[T_FIX] = -1;
                break;
            }
        } while ((int)(seen - target) < 0);
    }
    __syncthreads();
}
__device__ __forceinline__ double get_part_ll(const KRArgs &A, int which, int c, unsigned ll_epoch) {
    const unsigned long long *p = A.ll + 2 * ((int64_t)which * A.n_chunks + c);
    unsigned long long a, b;
    const long long t0 = clock64();
    do {
        asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
        if (A.n_rank > 1 && clock64() - t0 > A.peer_timeout) return __longlong_as_double(0x7ff8000000000000LL);
    } while ((unsigned)(a >> 32) != ll_epoch || (unsigned)(b >> 32) != ll_epoch);
    return __longlong_as_double((long long)((a & 0xffffffffull) | (b << 32)));
}

struct SpmvState {             // carried from tile to tile by the stitching warps
    double open;               // sum so far of the segment open at the end of the last tile
    int seen, last_ord;        // a segment start was seen in this CTA's range; ordinal of the latest one
};

static_assert(sizeof(SpmvState) == 16, "SM_STATE holds SpmvState followed by the CTA's 8-byte SpMV cycle counter");

struct Smem {
    double *red, *u;
    WarpRecs *rec;
    KRScalars *ctl;
    SpmvState *st;
    int *slab;
    uint64_t *mbar;
    unsigned u_phase;          // parity of the next completion of mbar
};

__device__ __forceinline__ Smem carve_smem(unsigned char *base) {
    Smem s;
    s.red = (double *)(base + SM_RED);
    s.rec = (WarpRecs *)(base + SM_REC);
    s.ctl = (KRScalars *)(base + SM_CTL);
    s.st = (SpmvState *)(base + SM_STATE);
    s.slab = (int *)(base + SM_SLAB);
    s.mbar = (uint64_t *)(base + SM_MBAR);
    s.u = (double *)(base + SM_U);
    s.u_phase = 0;
    return s;
}

// ---- TMA bulk copy + mbarrier (the u slab) ------------------------------------------------------
__device__ __forceinline__ unsigned smem_addr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *mbar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(mbar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *mbar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(mbar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *mbar, unsigned parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "B3C_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra B3C_DONE;\n\t"
        "bra B3C_WAIT;\n\t"
        "B3C_DONE:\n\t"
        "}" ::"r"(smem_addr(mbar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gsrc, unsigned bytes, uint64_t *mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_addr(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_addr(mbar))
                 : "memory");
}

// ---- deterministic block reductions ---------------------------------------------------------
// NS sums followed by NM minima, reduced together: warp xor-tree, then the warp results in warp
// order.  The results are valid in THREAD 0 only (every caller hands them to thread 0: a partial to
// publish, or the loop scalars); the shape is fixed, so the value is reproducible.
template <int NS, int NM>
__device__ __forceinline__ void block_reduce(double (&v)[NS + NM], double *s_red) {
    constexpr int K = NS + NM;
    static_assert(K <= RED_MAX, "too many values");
#pragma unroll
    for (int i = 0; i < K; ++i) v[i] = (i < NS) ? warp_sum(v[i]) : warp_min(v[i]);
    const unsigned w = threadIdx.x >> 5;
    __syncthreads();
    if (lane_id() == 0) {
#pragma unroll
        for (int i = 0; i < K; ++i) s_red[w * K + i] = v[i];
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        // lane i folds value i over the warps, in warp order (the K chains run side by side), then hands it to thread 0
        const int i = (int)lane_id() < K ? (int)lane_id() : 0;
        const bool is_sum = i < NS;
        double r = s_red[i];
#pragma unroll
        for (int j = 1; j < KR_WARPS; ++j) {
            const double x = s_red[j * K + i];
            const double a = r + x, m = fmin(r, x);
            r = is_sum ? a : m;
        }
#pragma unroll
        for (int k = 0; k < K; ++k) v[k] = __shfl_sync(kFullMask, r, k);
    }
}

// the same over per-chunk partial arrays: out[i] = reduce(part[ids[i]][0..nc)) in thread 0; identical in every CTA.
// Bit i of `ll_mask` set: partial ids[i] comes through the flagged words of epoch `ll_epoch` (see put_part).
template <int NS, int NM>
__device__ __forceinline__ void reduce_parts(const KRArgs &A, int nc, const int (&ids)[NS + NM],
                                             double (&out)[NS + NM], double *s_red, unsigned ll_mask = 0,
                                             unsigned ll_epoch = 0) {
    const double *part = A.part;
    if (ll_mask) ll_wait(A, ll_epoch * (unsigned)nc);         // every chunk arrives once per hand-over
#pragma unroll
    for (int i = 0; i < NS + NM; ++i) out[i] = (i < NS) ? 0.0 : (double)INFINITY;
    for (int j = threadIdx.x; j < nc; j += KR_THREADS) {
#pragma unroll
        for (int i = 0; i < NS + NM; ++i) {
            const double x = ((ll_mask >> i) & 1u) ? get_part_ll(A, ids[i], j, ll_epoch)
                                                   : __ldcg(part + (int64_t)ids[i] * nc + j);
            out[i] = (i < NS) ? out[i] + x : fmin(out[i], x);
        }
    }
    block_reduce<NS, NM>(out, s_red);
}

// ---- SpMV -------------------------------------------------------------------------------------
// Inside a 512-entry chunk lane l owns the 16 consecutive entries [16 l, 16 l + 16), and the chunk is STORED
// piece-major -- physical position k * 256 + 8 l + i holds logical entry 16 l + 8 k + i -- so the two
// pieces (k = 0, 1) of a chunk are each read with fully coalesced 64-byte-per-lane loads.
__host__ __device__ __forceinline__ int64_t stream_phys(int64_t logical) {
    const int64_t r = logical & (SPMV_CHUNK - 1);
    return (logical - r) + ((r >> 3) & 1) * (SPMV_CHUNK / 2) + (r >> 4) * SPMV_EPP + (r & 7);
}

// What a lane holds for one piece, loaded SPMV_DEPTH pieces ahead of its use.
struct PieceRegs {
    double a[SPMV_EPP];        // fp64 stream: the values
    unsigned long long q[SPMV_EPP / 2];   // counts stream: the eight uint32 counts, two per word
    unsigned c[SPMV_EPP];      // slab form: c[0..3] hold the 8 columns, 16 bit each; gather form: one column each
    unsigned fw;               // first piece of a chunk only: start flags of the lane's 16 entries
    int seg0;                  // first piece only: ordinal of the first segment that starts inside the chunk
};

template <bool SLAB, int CNT>
__device__ __forceinline__ void piece_load(const KRArgs &A, int64_t p, int64_t p_hi, PieceRegs &R) {
    if (p >= p_hi) return;
    const int64_t chunk = p >> 1;
    const int64_t e = chunk * SPMV_CHUNK + (p & 1) * (SPMV_CHUNK / 2) + SPMV_EPP * lane_id();
    if (CNT) {
        // eight uint32 counts -- or, packed form, eight (count << 16 | column) words -- in one 32-byte load, widened when
        // the piece is processed
        asm volatile("ld.global.nc.L1::no_allocate.v4.u64 {%0,%1,%2,%3}, [%4];"
                     : "=l"(R.q[0]), "=l"(R.q[1]), "=l"(R.q[2]), "=l"(R.q[3])
                     : "l"((const uint32_t *)A.sval + e));
    } else {
        asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];"
                     : "=d"(R.a[0]), "=d"(R.a[1]), "=d"(R.a[2]), "=d"(R.a[3])
                     : "l"(A.sval + e));
        asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];"
                     : "=d"(R.a[4]), "=d"(R.a[5]), "=d"(R.a[6]), "=d"(R.a[7])
                     : "l"(A.sval + e + 4));
    }
    if (CNT == 2) {
        // the columns came with the counts
    } else if (SLAB) {
        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(R.c[0]), "=r"(R.c[1]), "=r"(R.c[2]), "=r"(R.c[3])
                     : "l"((const uint16_t *)A.scol + e));
    } else {
        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(R.c[0]), "=r"(R.c[1]), "=r"(R.c[2]), "=r"(R.c[3])
                     : "l"((const uint32_t *)A.scol + e));
        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(R.c[4]), "=r"(R.c[5]), "=r"(R.c[6]), "=r"(R.c[7])
                     : "l"((const uint32_t *)A.scol + e + 4));
    }
    if ((p & 1) == 0) {
        unsigned short fw;
        asm volatile("ld.global.nc.L1::no_allocate.u16 %0, [%1];" : "=h"(fw) : "l"(A.sflag + chunk * 32 + lane_id()));
        R.fw = fw;
        R.seg0 = __ldg(A.chunk_seg0 + chunk);
    }
}

// L2 prefetch of the stream `dist` chunks ahead of the chunk a warp is about to process (KR_OPT_L2_PREFETCH: 6 chunks,
// + KR_OPT_L2_PREFETCH_FAR: 12 more): the register ring covers ~1.5 chunks, less than the DRAM latency under load --
// the SpMV's largest stall was the wait for a piece's own load -- so the ring's loads should find their lines in L2.
template <bool SLAB, int CNT>
__device__ __forceinline__ void chunk_prefetch(const KRArgs &A, int64_t chunk, int64_t chunk_hi) {
    if (chunk >= chunk_hi || lane_id() != 0) return;
    const char *v = (const char *)A.sval + chunk * SPMV_CHUNK * (CNT ? 4 : 8);
    const char *c = (const char *)A.scol + chunk * SPMV_CHUNK * (SLAB ? 2 : 4);
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(v), "r"(SPMV_CHUNK * (CNT ? 4 : 8)) : "memory");
    if (CNT != 2) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(c), "r"(SPMV_CHUNK * (SLAB ? 2 : 4)) : "memory");
}

// bring slab `slab` of u into shared memory: one thread issues TMA bulk copies, everybody waits on the mbarrier
__device__ __forceinline__ void slab_fetch(const KRArgs &A, const double *u, int slab, Smem &sm) {
    const int col0 = slab * A.W;
    int cnt = A.n - col0;
    if (cnt > A.W) cnt = A.W;
    const unsigned bytes = (unsigned)((cnt + 1) & ~1) * 8u;          // whole 16-byte units (the vectors are padded)
    if (threadIdx.x == 0) {
        asm volatile("fence.proxy.async;" ::: "memory");             // u was written through the generic proxy
        mbar_expect_tx(sm.mbar, bytes);
        constexpr unsigned PIECE = 32768;
        for (unsigned off = 0; off < bytes; off += PIECE)
            bulk_g2s((char *)sm.u + off, (const char *)(u + col0) + off, bytes - off < PIECE ? bytes - off : PIECE,
                     sm.mbar);
    }
    mbar_wait(sm.mbar, sm.u_phase);
    sm.u_phase ^= 1u;
}

// what a warp carries along its run of chunks (identical in all lanes)
struct WarpRun {
    double open;               // sum so far of the segment open at the end of the last chunk
    double head;               // sum of the entries before the run's first flag
    int seen, last;            // a segment start was seen; ordinal of the latest one
};
// what a lane carries through the pieces of a chunk
struct LaneRun {
    double cur, head;          // sum of the segment open at this point of the lane's run; sum before its first flag
    unsigned fw;               // flags not yet consumed
    int base, nseen;           // ordinal of the first segment starting in the lane's run; starts seen so far
    int lower, total, seg0;    // flags in lower lanes / in the whole chunk; the chunk's first ordinal
};

// One piece: 8 products per lane, added to the lane's running segment; a start flag closes the open segment.
template <bool SLAB, int CNT>
__device__ __forceinline__ void piece_process(const KRArgs &A, const double *u, const PieceRegs &R, const Smem &sm,
                                              bool first_piece, LaneRun &L) {
    const unsigned lane = lane_id();
    if (first_piece) {
        // segments start only at piece boundaries (seg_padded), so a lane's 16 entries carry at most two flags,
        // bits 0 and 8: the prefix count over the lanes is two ballots instead of a shuffle scan
        const unsigned f0 = __ballot_sync(kFullMask, (R.fw & 1u) != 0);
        const unsigned f1 = __ballot_sync(kFullMask, (R.fw & 0x100u) != 0);
        const unsigned lt = lanemask_lt();
        L.lower = __popc(f0 & lt) + __popc(f1 & lt);
        L.total = __popc(f0) + __popc(f1);
        L.seg0 = R.seg0;
        L.base = R.seg0 + L.lower;
        L.fw = R.fw;
        L.cur = 0.0;
        L.head = 0.0;
        L.nseen = 0;
    }
    double x[SPMV_EPP], a[SPMV_EPP];
    if (CNT == 2) {
        const double *su = sm.u;
#pragma unroll
        for (int i = 0; i < SPMV_EPP; ++i) {
            const uint32_t w = (uint32_t)(R.q[i >> 1] >> ((i & 1) * 32));
            x[i] = __dmul_rn((double)(w >> 16), su[w & 0xffffu]);
        }
    } else {
#pragma unroll
    for (int i = 0; i < SPMV_EPP; ++i)
        a[i] = CNT ? (double)(uint32_t)(R.q[i >> 1] >> ((i & 1) * 32)) : R.a[i];
    if (SLAB) {
        const double *su = sm.u;
#pragma unroll
        for (int i = 0; i < SPMV_EPP / 2; ++i) {
            x[2 * i] = __dmul_rn(a[2 * i], su[R.c[i] & 0xffffu]);
            x[2 * i + 1] = __dmul_rn(a[2 * i + 1], su[R.c[i] >> 16]);
        }
    } else {
#pragma unroll
        for (int i = 0; i < SPMV_EPP; ++i) x[i] = __dmul_rn(a[i], u[R.c[i]]);
    }
    }
    // segments are padded to whole pieces (seg_padded), so only the piece's first entry can carry a flag:
    // add the piece up as a fixed tree, then either extend the open segment or close it and open the next
    static_assert(SPMV_EPP == 8, "piece sum tree");
    const double s8 = __dadd_rn(__dadd_rn(__dadd_rn(x[0], x[1]), __dadd_rn(x[2], x[3])),
                                __dadd_rn(__dadd_rn(x[4], x[5]), __dadd_rn(x[6], x[7])));
    const unsigned bits = L.fw & 1u;
    L.fw >>= 8;
    if (bits) {
        if (L.nseen == 0) L.head = L.cur;
        else A.qs[L.base + L.nseen - 1] = L.cur;
        L.nseen += 1;
        L.cur = s8;
    } else {
        L.cur = __dadd_rn(L.cur, s8);
    }
}

// End of a chunk: stitch the 32 lane runs together (one segmented scan) and carry the open segment on.
__device__ __forceinline__ void chunk_finish(const KRArgs &A, const LaneRun &L, WarpRun &run) {
    const unsigned lane = lane_id();
    if (L.total == 0) {                                // the whole chunk continues the open segment
        run.open = __dadd_rn(run.open, warp_sum(L.cur));
        return;
    }
    const bool seen = L.nseen > 0;
    const unsigned any = __ballot_sync(kFullMask, seen);
    const unsigned lt = lanemask_lt();
    const unsigned le = any & (lt | (1u << lane));
    const int start = le ? 31 - __clz(le) : 0;         // nearest lane at or below me holding a flag
    double V = L.cur;                                  // lane sum since its last flag (all 16 entries if it has none)
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(kFullMask, V, o);
        if ((int)lane - o >= start) V = __dadd_rn(t, V);
    }
    double Oprev = __shfl_up_sync(kFullMask, V, 1);    // sum of the segment open at the end of the lane below
    if (lane == 0) Oprev = 0.0;
    const double closing = __dadd_rn(Oprev, L.head);   // the segment open at my start ends at my first flag
    if (seen && L.lower > 0) A.qs[L.base - 1] = closing;
    // the lane holding the chunk's first flag closes the run's open segment
    const double chead = __shfl_sync(kFullMask, closing, __ffs(any) - 1);
    const double rclose = __dadd_rn(run.open, chead);
    if (!run.seen) run.head = rclose;
    else if (lane == 0) A.qs[L.seg0 - 1] = rclose;
    run.open = __shfl_sync(kFullMask, V, 31);
    run.seen = 1;
    run.last = L.seg0 + L.total - 1;
}

// One warp stitches the runs of the 16 warps over a part of the CTA's range: closes the segment that was
// open when a run with flags began, carries the open segment forward, and writes the CTA's boundary
// record after the last part.
__device__ __forceinline__ void part_stitch(const KRArgs &A, const Smem &sm, int buf, bool last_part) {
    const unsigned lane = lane_id();
    const bool act = lane < KR_WARPS;
    const WarpRecs &rec = sm.rec[buf];
    const double head = act ? rec.head[lane] : 0.0;
    const double tail = act ? rec.tail[lane] : 0.0;
    const int seen = act ? rec.seen[lane] : 0;
    const int first = act ? rec.first[lane] : 0;
    const int lastv = act ? rec.last[lane] : 0;
    const double open_in = sm.st->open;
    const int seen_in = sm.st->seen;
    int last_ord = sm.st->last_ord;
    __syncwarp();
    const unsigned fm = __ballot_sync(kFullMask, seen != 0);
    const unsigned lt = lanemask_lt();
    const unsigned le = fm & (lt | (1u << lane));
    const int start = le ? 31 - __clz(le) : 0;
    double V = seen ? tail : head;
#pragma unroll
    for (int o = 1; o < KR_WARPS; o <<= 1) {
        const double t = __shfl_up_sync(kFullMask, V, o);
        if ((int)lane - o >= start) V = __dadd_rn(t, V);
    }
    const double O = le ? V : __dadd_rn(open_in, V);               // open sum after warp `lane`'s run
    double Oprev = __shfl_up_sync(kFullMask, O, 1);
    if (lane == 0) Oprev = open_in;
    if (act && seen) {
        const double closing = __dadd_rn(Oprev, head);
        if (!seen_in && !(fm & lt)) A.bnd_head[blockIdx.x] = closing;  // the CTA's first flag: closes its head
        else A.qs[first - 1] = closing;
    }
    const double open_out = __shfl_sync(kFullMask, O, KR_WARPS - 1);
    if (fm) last_ord = __shfl_sync(kFullMask, lastv, 31 - __clz(fm));
    if (lane == 0) {
        sm.st->open = open_out;
        sm.st->seen = seen_in | (fm != 0);
        sm.st->last_ord = last_ord;
        if (last_part) {
            const int b = blockIdx.x;
            if (seen_in | (fm != 0)) {
                A.bnd_tail[b] = open_out;
                A.bnd_ord[b] = last_ord;
                A.bnd_lr[b] = __ldg(A.seg_row + last_ord) % A.npad;
                A.bnd_flag[b] = 1;
            } else {
                A.bnd_head[b] = open_out;
                A.bnd_flag[b] = 0;
            }
        }
    }
}

// The SpMV phase.  The CTA owns a contiguous range of chunks; it is cut into parts at slab boundaries
// (almost always one part), and inside a part every warp streams its own contiguous run of chunks with no
// block-wide synchronisation; the runs are stitched once per part.
template <bool SLAB, int CNT>
__device__ __forceinline__ void phase_spmv(const KRArgs &A, const double *u, Smem &sm) {
    for (int i = threadIdx.x; i <= A.S; i += KR_THREADS) sm.slab[i] = A.slab_c0[i];
    if (threadIdx.x == 0) {
        sm.st->open = 0.0;
        sm.st->seen = 0;
        sm.st->last_ord = -1;
    }
    __syncthreads();
    int64_t c_lo = A.n_sch * blockIdx.x / gridDim.x, c_hi = A.n_sch * (blockIdx.x + 1) / gridDim.x;
    if (SLAB && (A.opts & KR_OPT_SLAB_ALIGN) && A.S > 1 && (int)gridDim.x >= 2 * A.S) {
        // CTA ranges follow the slabs: every slab gets a share of the grid proportional to its chunks, so no
        // CTA fetches two slabs of u (a range straddling a slab boundary would, and hold the grid barrier up)
        const int G = gridDim.x, g = blockIdx.x;
        int b_lo = 0, b_hi = G, s_mine = 0, prev = 0;
        for (int k = 0; k < A.S; ++k) {
            int nxt = G;
            if (k + 1 < A.S) {
                nxt = (int)(((int64_t)sm.slab[k + 1] * G + A.n_sch / 2) / A.n_sch);
                if (nxt < prev + 1) nxt = prev + 1;
                if (nxt > G - (A.S - 1 - k)) nxt = G - (A.S - 1 - k);
            }
            if (g >= prev && g < nxt) {
                s_mine = k;
                b_lo = prev;
                b_hi = nxt;
            }
            prev = nxt;
        }
        const int64_t s0 = sm.slab[s_mine], len = sm.slab[s_mine + 1] - s0;
        c_lo = s0 + len * (g - b_lo) / (b_hi - b_lo);
        c_hi = s0 + len * (g - b_lo + 1) / (b_hi - b_lo);
    }
    if (c_lo >= c_hi) {
        if (threadIdx.x == 0) {
            A.bnd_head[blockIdx.x] = 0.0;
            A.bnd_flag[blockIdx.x] = 0;
        }
        __syncthreads();
        return;
    }
    const int warp = threadIdx.x >> 5;
    int slab = 0, part = 0;
    for (int64_t p_lo = c_lo; p_lo < c_hi; ++part) {
        while (p_lo >= sm.slab[slab + 1]) ++slab;
        const int64_t slab_end = sm.slab[slab + 1];
        const int64_t p_hi = slab_end < c_hi ? slab_end : c_hi;
        const int64_t n = p_hi - p_lo;
        const int64_t w_lo = p_lo + n * warp / KR_WARPS, w_hi = p_lo + n * (warp + 1) / KR_WARPS;
        const int64_t q_lo = 2 * w_lo, q_hi = 2 * w_hi;            // pieces
        PieceRegs R0, R1, R2;
        piece_load<SLAB, CNT>(A, q_lo, q_hi, R0);
        piece_load<SLAB, CNT>(A, q_lo + 1, q_hi, R1);
        piece_load<SLAB, CNT>(A, q_lo + 2, q_hi, R2);
        // every gather of the previous part is behind that part's barrier, so the slab can be replaced
        if (SLAB) slab_fetch(A, u, slab, sm);
        WarpRun run;
        run.open = 0.0;
        run.head = 0.0;
        run.seen = 0;
        run.last = -1;
        LaneRun L;
        L.cur = L.head = 0.0;
        L.fw = 0;
        L.base = L.nseen = L.lower = L.total = L.seg0 = 0;
        int first = 0;
        if (q_lo < q_hi) first = R0.seg0;
        // the ring has three stages and a chunk two pieces: six pieces (three chunks) per trip keep every index static
        const int pf_dist = ((A.opts & KR_OPT_L2_PREFETCH) ? 6 : 0) + ((A.opts & KR_OPT_L2_PREFETCH_FAR) ? 12 : 0);
        if (pf_dist)
            for (int d = 2; d < pf_dist; ++d) chunk_prefetch<SLAB, CNT>(A, w_lo + d, w_hi);
        for (int64_t q = q_lo; q < q_hi; q += 6) {
            if (pf_dist) {
                const int64_t ck = (q >> 1) + pf_dist;
                chunk_prefetch<SLAB, CNT>(A, ck, w_hi);
                chunk_prefetch<SLAB, CNT>(A, ck + 1, w_hi);
                chunk_prefetch<SLAB, CNT>(A, ck + 2, w_hi);
            }
            piece_process<SLAB, CNT>(A, u, R0, sm, true, L);
            piece_load<SLAB, CNT>(A, q + 3, q_hi, R0);
            piece_process<SLAB, CNT>(A, u, R1, sm, false, L);
            piece_load<SLAB, CNT>(A, q + 4, q_hi, R1);
            chunk_finish(A, L, run);
            if (q + 2 < q_hi) {
                piece_process<SLAB, CNT>(A, u, R2, sm, true, L);
                piece_load<SLAB, CNT>(A, q + 5, q_hi, R2);
                piece_process<SLAB, CNT>(A, u, R0, sm, false, L);
                piece_load<SLAB, CNT>(A, q + 6, q_hi, R0);
                chunk_finish(A, L, run);
            }
            if (q + 4 < q_hi) {
                piece_process<SLAB, CNT>(A, u, R1, sm, true, L);
                piece_load<SLAB, CNT>(A, q + 7, q_hi, R1);
                piece_process<SLAB, CNT>(A, u, R2, sm, false, L);
                piece_load<SLAB, CNT>(A, q + 8, q_hi, R2);
                chunk_finish(A, L, run);
            }
        }
        if (lane_id() == 0) {
            WarpRecs &rec = sm.rec[part & 1];
            rec.head[warp] = run.seen ? run.head : run.open;
            rec.tail[warp] = run.open;
            rec.seen[warp] = run.seen;
            rec.first[warp] = first;
            rec.last[warp] = run.last;
        }
        __syncthreads();
        if (warp == part % KR_WARPS) part_stitch(A, sm, part & 1, p_hi == c_hi);
        p_lo = p_hi;
    }
    __syncthreads();                   // the next phase reuses the shared-memory reduction scratch
}

// Finish the segments that cross SpMV CTA ranges: the segment open at the end of CTA g's range is
// its tail plus the heads of the following CTAs up to (and including) the first one that saw a flag.
// The CTA that owns reduction chunk c does this for the rows of the chunk before it reads their sums.
// Everything a record can need in the common case (its own fields and the next CTA's head and flag) is
// loaded up front, so the fix costs one trip to L2 instead of a chain of three or four.
__device__ __forceinline__ void boundary_fix(const KRArgs &A, int c) {
    const int64_t r0 = (int64_t)c * CHUNK - A.row_lo;              // local rows [r0, r0 + CHUNK)
    for (int g = threadIdx.x; g < A.n_bnd; g += KR_THREADS) {
        const bool nxt = g + 1 < A.n_bnd;
        const int flag = __ldcg(A.bnd_flag + g);
        const int lr = __ldcg(A.bnd_lr + g);
        const int ord = __ldcg(A.bnd_ord + g);
        double s = __ldcg(A.bnd_tail + g);
        const double h1 = nxt ? __ldcg(A.bnd_head + g + 1) : 0.0;
        const int f1 = nxt ? __ldcg(A.bnd_flag + g + 1) : 1;
        if (!flag || lr < r0 || lr >= r0 + CHUNK) continue;
        if (nxt) {
            s = __dadd_rn(s, h1);
            if (!f1) {
                for (int g2 = g + 2; g2 < A.n_bnd; ++g2) {
                    s = __dadd_rn(s, __ldcg(A.bnd_head + g2));
                    if (__ldcg(A.bnd_flag + g2)) break;
                }
            }
        }
        A.qs[ord] = s;
    }
    __syncthreads();
}

// (A u)[r]: the segment sums of global row r, added in slab order (loads batched eight slabs at a time)
__device__ __forceinline__ double row_q(const KRArgs &A, int64_t r) {
    const int64_t lr = r - A.row_lo;
    double s = 0.0;
    for (int k0 = 0; k0 < A.S; k0 += 8) {
        int o[8];
        double t[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] = k0 + k < A.S ? __ldg(A.seg_of + (int64_t)(k0 + k) * A.npad + lr) : -1;
#pragma unroll
        for (int k = 0; k < 8; ++k) t[k] = o[k] >= 0 ? __ldcg(A.qs + o[k]) : 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (o[k] >= 0) s = __dadd_rn(s, t[k]);
    }
    return s;
}

// ---- vector phases: one CTA per 1024-row chunk, CHUNK_RPT rows per thread ------------------------
// Every phase first LOADS what its CHUNK_RPT rows need (independent L2 reads, issued back to back), then computes
// and stores: the vectors are rewritten from phase to phase, so they are read with ld.global.cg (L2) and a
// store can never force a later load to wait.
#define KR_FOR_CHUNKS(c) for (int c = blockIdx.x; c < A.n_chunks; c += gridDim.x)
#define KR_ROW(c, i) ((int64_t)(c) * CHUNK + (i) * KR_THREADS + threadIdx.x)
constexpr int ROWQ_S = 12;                     // slabs per round of the batched rows_q

__device__ __forceinline__ bool chunk_local(const KRArgs &A, int c) {
    const int64_t r0 = (int64_t)c * CHUNK;
    return r0 >= A.row_lo && r0 < A.row_hi;
}

// Packed count stream: the high parts of row r's off-diagonal counts above 65535 (side list sorted by row, then
// column) times the scaled operand, added to the row sum in list order
__device__ __forceinline__ double add_big(const KRArgs &A, int64_t r, double s, const double *mult) {
    int lo = 0, hi = A.n_big;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(A.big_row + mid) < (int32_t)r) lo = mid + 1;
        else hi = mid;
    }
    for (; lo < A.n_big && __ldg(A.big_row + lo) == (int32_t)r; ++lo)
        s = __dadd_rn(s, __dmul_rn(__ldg(A.big_hi + lo), __ldcg(mult + __ldg(A.big_col + lo))));
    return s;
}

// q = A u plus the zero-diagonal term (Q2) for the CHUNK_RPT rows of this thread, loads batched: every cell
// ordinal of NB slabs (of all the thread's rows) first, then every segment sum, then the adds in slab order; matrices
// wider than NB slabs take several such rounds (C4's 35 slabs: 3 rounds of 2 dependent trips instead of the 20 a
// row-by-row walk in batches of eight took -- the vector phases of a wide matrix are latency-bound)
template <int NB, bool MULTI>
__device__ __forceinline__ void rows_q_batched(const KRArgs &A, const double *opnd, int c, double (&qq)[CHUNK_RPT]) {
    int o[CHUNK_RPT][NB];
    double df[CHUNK_RPT], uu[CHUNK_RPT], is[CHUNK_RPT], t[CHUNK_RPT][NB], s[CHUNK_RPT];
    bool ok[CHUNK_RPT];
#pragma unroll
    for (int i = 0; i < CHUNK_RPT; ++i) {
        const int64_t r = KR_ROW(c, i);
        ok[i] = r < A.row_hi;
#pragma unroll
        for (int k = 0; k < NB; ++k)
            o[i][k] = (ok[i] && k < A.S) ? __ldg(A.seg_of + (int64_t)k * A.npad + (r - A.row_lo)) : -1;
        df[i] = ok[i] ? __ldcg(A.dfix + r) : 0.0;
        uu[i] = ok[i] ? __ldcg(opnd + r) : 0.0;
        is[i] = (ok[i] && A.cnt_stream) ? __ldg(A.inv_s + r) : 1.0;
        s[i] = 0.0;
    }
    for (int k0 = 0;;) {
#pragma unroll
        for (int i = 0; i < CHUNK_RPT; ++i)
#pragma unroll
            for (int k = 0; k < NB; ++k) t[i][k] = o[i][k] >= 0 ? __ldcg(A.qs + o[i][k]) : 0.0;
#pragma unroll
        for (int i = 0; i < CHUNK_RPT; ++i)
#pragma unroll
            for (int k = 0; k < NB; ++k)
                if (o[i][k] >= 0) s[i] = __dadd_rn(s[i], t[i][k]);
        if constexpr (MULTI) {
            k0 += NB;
            if (k0 >= A.S) break;
#pragma unroll
            for (int i = 0; i < CHUNK_RPT; ++i) {
                const int64_t r = KR_ROW(c, i);
#pragma unroll
                for (int k = 0; k < NB; ++k)
                    o[i][k] = (ok[i] && k0 + k < A.S) ? __ldg(A.seg_of + (int64_t)(k0 + k) * A.npad + (r - A.row_lo)) : -1;
            }
        } else {
            break;
        }
    }
#pragma unroll
    for (int i = 0; i < CHUNK_RPT; ++i) {
        double q = s[i];
        if (__double_as_longlong(df[i]) < 0) {                    // the side list names this row (sign bit of dfix)
            q = add_big(A, KR_ROW(c, i), q, opnd == A.u ? A.us : A.xs);
            df[i] = fabs(df[i]);
        }
        if (A.cnt_stream) q = __dmul_rn(q, is[i]);                 // counts stream: the row's 1 / s_i
        if (df[i] != 0.0) q = __dadd_rn(q, __dmul_rn(df[i], uu[i]));   // zero diagonal counted as one (Q2): df = 1; or the
                                                                    // high part of a packed diagonal count (KRArgs.cnt_stream)
        qq[i] = q;
    }
}

// `opnd`: the vector the SpMV just multiplied (u, or x for a residual), for the zero-diagonal term
__device__ __forceinline__ void rows_q(const KRArgs &A, const double *opnd, int c, double (&qq)[CHUNK_RPT]) {
    if (A.S <= 4) return rows_q_batched<4, false>(A, opnd, c, qq);
    if (A.S <= ROWQ_S) return rows_q_batched<ROWQ_S, false>(A, opnd, c, qq);
    return rows_q_batched<ROWQ_S, true>(A, opnd, c, qq);
}

__device__ __forceinline__ void phase_init(const KRArgs &A) {
    KR_FOR_CHUNKS(c) {
        if (!chunk_local(A, c)) continue;
#pragma unroll
        for (int i = 0; i < CHUNK_RPT; ++i) {
            const int64_t r = KR_ROW(c, i);
            if (r < A.row_hi) {
                A.x[r] = 1.0;
                put_u(A, r, 1.0);
            }
        }
    }
}

// persistent kernel: x = 1 on the rows of this rank, published to every rank (the first SpMV multiplies x itself)
__device__ __forceinline__ void phase_init_p(const KRArgs &A) {
    KR_FOR_CHUNKS(c) {
        if (!chunk_local(A, c)) continue;
#pragma unroll
        for (int i = 0; i < CHUNK_RPT; ++i) {
            const int64_t r = KR_ROW(c, i);
            if (r < A.row_hi) put_x(A, r, 1.0);
        }
    }
}

// v = x * (A x), rk = 1 - v, partial rk.rk           (sparse_utils.py:136-139, 196-199)
// and -- used only if an inner loop follows -- Z = rk / v of its first CG step with the partial rk.Z (Q1,
// sparse_utils.py:158-160), published with the residual's own hand-over.  `opnd` is what the SpMV multiplied.
__device__ __forceinline__ void phase_resid(const KRArgs &A, const double *opnd, double *s_red, unsigned ll = 0) {
    KR_FOR_CHUNKS(c) {
        double acc = 0.0, accz = 0.0;
        const bool loc = chunk_local(A, c);
        if (!loc && A.n_rank > 1) continue;            // peer mode: the owner of a chunk publishes its partials
        if (loc) {
            double xx[CHUNK_RPT], qq[CHUNK_RPT];
#pragma unroll
            for (int i = 0; i < CHUNK_RPT; ++i) {
                const int64_t r = KR_ROW(c, i);
                xx[i] = r < A.row_hi ? __ldcg(A.x + r) : 0.0;
            }
            boundary_fix(A, c);
            rows_q(A, opnd, c, qq);
#pragma unroll
            for (int i = 0; i < CHUNK_RPT; ++i) {
                const int64_t r = KR_ROW(c, i);
                if (r < A.row_hi) {
                    const double vv = __dmul_rn(xx[i], qq[i]);
                    const double rr = __dsub_rn(1.0, vv);
                    A.v[r] = vv;
                    A.rk[r] = rr;
                    acc = __dadd_rn(acc, __dmul_rn(rr, rr));
                    const double z = __ddiv_rn(rr, vv);                       // sparse_utils.py:158
                    put_z(A, r, z);
                    accz = __dadd_rn(accz, __dmul_rn(rr, z));
                }
            }
        }
        double r[2] = {acc, accz};
        block_reduce<2, 0>(r, s_red);
        if (threadIdx.x == 0) {
            put_part(A, PB, c, r[1], loc, 0.0);
            put_part(A, PA, c, r[0], loc, 0.0, ll);
            if (ll) ll_arrive(A);
        }
    }
}

// persistent kernel: the direction of a CG step for ALL rows, on every rank (x and Z are complete everywhere, p is
// kept for all rows): first step p = Z (sparse_utils.py:159), later steps p = Z + beta p (:163); u = x * p.  No data
// leaves the GPU, so the phase ends with a local grid barrier.
__device__ __forceinline__ void phase_dir_all(const KRArgs &A, bool first, double beta, double *ycur) {
    KR_FOR_CHUNKS(c) {
        const bool loc = chunk_local(A, c);
        double zz[CHUNK_RPT], pp[CHUNK_RPT], xx[CHUNK_RPT];
#pragma unroll
        for (int i = 0; i < CHUNK_RPT; ++i) {
            const int64_t r = KR_ROW(c, i);
            const bool ok = r < A.n;
            zz[i] = ok ? __ldcg(A.Z + r) : 0.0;
            pp[i] = (ok && !first) ? __ldcg(A.p + r) : 0.0;
            xx[i] = ok ? __ldcg(A.x + r) : 0.0;
        }
#pragma unroll
        for (int i = 0; i < CHUNK_RPT; ++i) {
            const int64_t r = KR_ROW(c, i);
            if (r < A.n) {
                const double pn = first ? zz[i] : __dadd_rn(zz[i], __dmul_rn(beta, pp[i]));
                A.p[r] = pn;
                const double un = __dmul_rn(xx[i], pn);
                A.u[r] = un;
                if (A.cnt_stream) A.us[r] = __dmul_rn(un, __ldg(A.inv_s + r));
                if (first && loc) ycur[r] = 1.0;                              // y[:] = e (sparse_utils.py:150)
            }
        }
    }
}

// first CG step: Z = rk / v, p = Z, partial rk.Z (Q1); later steps: p = Z + beta p.  u = x * p
__device__ __forceinline__ void phase_dir(const KRArgs &A, bool first, double beta, double *ycur, double *s_red) {
    KR_FOR_CHUNKS(c) {
        double acc = 0.0;
        const bool loc = chunk_local(A, c);
        if (loc) {
            double a0[CHUNK_RPT], a1[CHUNK_RPT], xx[CHUNK_RPT];
#pragma unroll
            for (int i = 0; i < CHUNK_RPT; ++i) {
                const int64_t r = KR_ROW(c, i);
                const bool ok = r < A.row_hi;
                a0[i] = ok ? __ldcg((first ? A.rk : A.Z) + r) : 0.0;
                a1[i] = ok ? __ldcg((first ? A.v : A.p) + r) : 1.0;
                xx[i] = ok ? __ldcg(A.x + r) : 0.0;
            }
#pragma unroll
            for (int i = 0; i < CHUNK_RPT; ++i) {
                const int64_t r = KR_ROW(c, i);
                if (r < A.row_hi) {
                    double pp;
                    if (first) {
                        const double z = __ddiv_rn(a0[i], a1[i]);           // sparse_utils.py:158
                        A.Z[r] = z;
                        pp = z;
                        acc = __dadd_rn(acc, __dmul_rn(a0[i], z));
                        ycur[r] = 1.0;                                      // y[:] = e (sparse_utils.py:150)
                    } else {
                        pp = __dadd_rn(a0[i], __dmul_rn(beta, a1[i]));      // sparse_utils.py:163
                    }
                    A.p[r] = pp;
                    put_u(A, r, __dmul_rn(xx[i], pp));
                }
            }
        }
        if (first) {
            double r[1] = {acc};
            block_reduce<1, 0>(r, s_red);
            if (threadIdx.x == 0) put_part(A, PB, c, r[0], loc, 0.0);
        } else if (threadIdx.x == 0) {
            put_part(A, PB, c, 0.0, loc, 0.0);
        }
    }
}

// w = x * (A (x p)) + v * p, partial p.w              (sparse_utils.py:165-166)
__device__ __forceinline__ void phase_w(const KRArgs &A, double *s_red, unsigned ll = 0) {
    KR_FOR_CHUNKS(c) {
        double acc = 0.0;
        const bool loc = chunk_local(A, c);
        if (!loc && A.n_rank > 1) continue;
        if (loc) {
            double xx[CHUNK_RPT], vv[CHUNK_RPT], pp[CHUNK_RPT], qq[CHUNK_RPT];
#pragma unroll
            for (int i = 0; i < CHUNK_RPT; ++i) {
                const int64_t r = KR_ROW(c, i);
                const bool ok = r < A.row_hi;
                xx[i] = ok ? __ldcg(A.x + r) : 0.0;
                vv[i] = ok ? __ldcg(A.v + r) : 0.0;
                pp[i] = ok ? __ldcg(A.p + r) : 0.0;
            }
            boundary_fix(A, c);
            rows_q(A, A.u, c, qq);
#pragma unroll
            for (int i = 0; i < CHUNK_RPT; ++i) {
                const int64_t r = KR_ROW(c, i);
                if (r < A.row_hi) {
                    const double ww = __dadd_rn(__dmul_rn(xx[i], qq[i]), __dmul_rn(vv[i], pp[i]));
                    A.w[r] = ww;
                    acc = __dadd_rn(acc, __dmul_rn(pp[i], ww));
                }
            }
        }
        double r[1] = {acc};
        block_reduce<1, 0>(r, s_red);
        if (threadIdx.x == 0) {
            put_part(A, PA, c, r[0], loc, 0.0, ll);
            if (ll) ll_arrive(A);
        }
    }
}

// ap = alpha p, ynew = y + ap, min/max and both clamp factors, and -- speculatively, used only if
// the step is accepted -- rk -= alpha w, Z = rk * v (Q1), partial rk.Z   (sparse_utils.py:167-190)
__device__ __forceinline__ void phase_step(const KRArgs &A, double alpha, double delta, double Delta,
                                           const double *ycur, double *ynew, double *s_red, unsigned ll = 0) {
    KR_FOR_CHUNKS(c) {
        double rho = 0.0, mn = INFINITY, nmx = INFINITY, g1 = INFINITY, g2 = INFINITY;
        const bool loc = chunk_local(A, c);
        if (!loc && A.n_rank > 1) continue;
        if (loc) {
            double pp[CHUNK_RPT], yv[CHUNK_RPT], rk[CHUNK_RPT], ww[CHUNK_RPT], vv[CHUNK_RPT];
#pragma unroll
            for (int i = 0; i < CHUNK_RPT; ++i) {
                const int64_t r = KR_ROW(c, i);
                const bool ok = r < A.row_hi;
                pp[i] = ok ? __ldcg(A.p + r) : 0.0;
                yv[i] = ok ? __ldcg(ycur + r) : 0.0;
                rk[i] = ok ? __ldcg(A.rk + r) : 0.0;
                ww[i] = ok ? __ldcg(A.w + r) : 0.0;
                vv[i] = ok ? __ldcg(A.v + r) : 0.0;
            }
#pragma unroll
            for (int i = 0; i < CHUNK_RPT; ++i) {
                const int64_t r = KR_ROW(c, i);
                if (r < A.row_hi) {
                    const double ap = __dmul_rn(alpha, pp[i]);
                    const double yy = yv[i];
                    const double yn = __dadd_rn(yy, ap);
                    ynew[r] = yn;
                    mn = fmin(mn, yn);
                    nmx = fmin(nmx, -yn);
                    if (ap < 0.0) g1 = fmin(g1, __ddiv_rn(__dsub_rn(delta, yy), ap));      // :174-175
                    if (yn > Delta) g2 = fmin(g2, __ddiv_rn(__dsub_rn(Delta, yy), ap));    // :180-181
                    const double rr = __dsub_rn(rk[i], __dmul_rn(alpha, ww[i]));          // :186
                    const double z = __dmul_rn(rr, vv[i]);                                // :189
                    A.rk[r] = rr;
                    put_z(A, r, z);
                    rho = __dadd_rn(rho, __dmul_rn(rr, z));
                }
            }
        }
        double r[5] = {rho, mn, nmx, g1, g2};
        block_reduce<1, 4>(r, s_red);
        if (threadIdx.x == 0) {
            put_part(A, PC, c, r[0], loc, 0.0, ll);
            put_part(A, PMIN, c, r[1], loc, (double)INFINITY, ll);
            put_part(A, PNEGMAX, c, r[2], loc, (double)INFINITY, ll);
            put_part(A, PG1, c, r[3], loc, (double)INFINITY, ll);
            put_part(A, PG2, c, r[4], loc, (double)INFINITY, ll);
            if (ll) ll_arrive(A);
        }
    }
}

// x *= y (y possibly clamped: y + gamma * alpha p), u = x      (sparse_utils.py:176,182,195)
template <bool PUBLISH_X>
__device__ __forceinline__ void phase_update(const KRArgs &A, int ymode, double gamma, double alpha,
                                             const double *ycur) {
    KR_FOR_CHUNKS(c) {
        if (!chunk_local(A, c)) continue;
        double xx[CHUNK_RPT], yv[CHUNK_RPT], pp[CHUNK_RPT];
#pragma unroll
        for (int i = 0; i < CHUNK_RPT; ++i) {
            const int64_t r = KR_ROW(c, i);
            const bool ok = r < A.row_hi;
            xx[i] = ok ? __ldcg(A.x + r) : 0.0;
            yv[i] = (ok && ymode >= 1) ? __ldcg(ycur + r) : 1.0;
            pp[i] = (ok && ymode == 2) ? __ldcg(A.p + r) : 0.0;
        }
#pragma unroll
        for (int i = 0; i < CHUNK_RPT; ++i) {
            const int64_t r = KR_ROW(c, i);
            if (r < A.row_hi) {
                double yy = yv[i];
                if (ymode == 2) yy = __dadd_rn(yy, __dmul_rn(gamma, __dmul_rn(alpha, pp[i])));
                const double xn = __dmul_rn(xx[i], yy);
                if (PUBLISH_X) {
                    put_x(A, r, xn);                   // persistent kernel: the next SpMV multiplies x itself
                } else {
                    A.x[r] = xn;
                    put_u(A, r, xn);
                }
            }
        }
    }
}

// ---- scalar logic ------------------------------------------------------------------------------------
// after a residual phase: rho = rk.rk; first call initialises, later calls close an outer step
__device__ __forceinline__ void scalar_outer(KRScalars &S, double rho, bool first) {
    const double g = 0.9, etamax = 0.1;
    S.rho_km1 = rho;
    S.rout = rho;
    if (first) {
        S.rold = rho;
        return;
    }
    S.n_iter += S.k + 1;                                  // sparse_utils.py:201
    const double rat = S.rout / S.rold;
    S.rold = S.rout;
    const double res_norm = sqrt(S.rout);
    const double eta_o = S.eta;
    S.eta = g * rat;
    if (g * eta_o * eta_o > 0.1) S.eta = fmax(S.eta, g * eta_o * eta_o);
    S.eta = fmax(fmin(S.eta, etamax), S.stop_tol / res_norm);
}

// after a step phase: accept or clamp.  returns true when the inner loop must stop.
__device__ __forceinline__ bool scalar_decide(KRScalars &S, double ymin, double ymax, double g1, double g2,
                                              double rho_new) {
    if (ymin <= S.delta) {                                // sparse_utils.py:171-177
        S.gamma = (S.delta == 0.0) ? 0.0 : g1;
        S.ymode = 2;
        return true;
    }
    if (ymax >= S.Delta) {                                // sparse_utils.py:179-183
        if (isinf(g2)) S.status = B3C_ERR_TIE;            // no element above Delta: exact tie (Q13)
        S.gamma = isinf(g2) ? 0.0 : g2;
        S.ymode = 2;
        return true;
    }
    S.ymode = 1;                                          // y = ynew
    S.ysel ^= 1;
    S.rho_km2 = S.rho_km1;
    S.rho_km1 = rho_new;
    return false;
}

// ---- loop control ------------------------------------------------------------------------------------
// One decision at a time on the reduced partials r[]; leaves the next thing to do in S.state.  Shared by the
// persistent kernel and the phase-at-a-time form (k_krp_scalar), so both take exactly the same branches.
enum { KRP_INIT = 0, KRP_SPMV, KRP_RESID, KRP_DIR, KRP_W, KRP_STEP, KRP_UPDATE };
enum { KRS_OUTER_FIRST = 0, KRS_OUTER, KRS_ALPHA, KRS_DECIDE };
enum { KR_STATE_DONE = 0, KR_STATE_INNER = 1, KR_STATE_UPDATE = 2 };

__device__ __forceinline__ void scalar_step(KRScalars &S, int which, const double *r) {
    if (which == KRS_OUTER_FIRST || which == KRS_OUTER) {          // r[0] = rk.rk
        scalar_outer(S, r[0], which == KRS_OUTER_FIRST);
        S.n_spmv += 1;
        if (isnan(S.rout)) S.status = B3C_ERR_NAN;                 // sparse_utils.py:192-193
        if (S.rout > S.rt && S.n_iter < S.max_iter) {              // sparse_utils.py:146
            S.outer += 1;
            S.k = 0;
            S.ymode = 0;
            S.inner_tol = fmax(S.rout * S.eta * S.eta, S.rt);
            if (S.rho_km1 > S.inner_tol) {                         // sparse_utils.py:154
                S.k = 1;
                S.state = KR_STATE_INNER;
            } else {
                S.state = KR_STATE_UPDATE;
            }
        } else {
            S.state = KR_STATE_DONE;
        }
    } else if (which == KRS_ALPHA) {                               // r[0] = p.w, r[1] = rk.Z of the first step
        if (S.k == 1) S.rho_km1 = r[1];                            // sparse_utils.py:160
        S.alpha = S.rho_km1 / r[0];                                // sparse_utils.py:166
        S.n_spmv += 1;
    } else if (which == KRS_DECIDE) {                              // r = rk.Z, min y, -max y, both clamp factors
        bool stop = scalar_decide(S, r[1], -r[2], r[3], r[4], r[0]);
        if (!stop && S.k >= S.max_iter + 8) {                      // safety net: the reference's inner loop is unbounded
            S.status = B3C_ERR_NOCONV;
            stop = true;
        }
        if (S.status != 0) {
            S.state = KR_STATE_DONE;
        } else if (stop) {
            S.state = KR_STATE_UPDATE;
        } else if (S.rho_km1 > S.inner_tol) {
            S.k += 1;
            S.beta = S.rho_km1 / S.rho_km2;
            S.state = KR_STATE_INNER;
        } else {
            S.state = KR_STATE_UPDATE;
        }
    }
}

// ---- the persistent kernel ---------------------------------------------------------------------------
// The loop scalars live in shared memory: thread 0 updates them between block barriers, everybody reads
// them; all CTAs compute identical values from the same partials.  One trip of the loop is
// "make u | SpMV | consume": init or update -> residual (an outer Newton step), direction -> w, step (a CG step).
// Barrier after a phase: one arrive counter + one generation word in global memory (the kernel is launched
// cooperatively, so all CTAs are resident).  Thread 0 of every CTA fences and arrives; the last CTA to
// arrive opens the next generation.  `cross`: the phase published data to the other GPUs -- the fences are
// system-wide, and before opening the generation the last CTA tells every rank this one has arrived
// (release store into its flag array over NVLink) and waits until all ranks have (acquire loads of the local
// flags).  A rank that never arrives (it failed before its launch) would hang the node, so that wait gives
// up after the peer time-out (B3C_OPT_PEER_TIMEOUT_MS, default 60 s) and poisons the local partials with NaN: every CTA then derives NaN scalars, the loop
// conditions fail, the kernel ends and the host reports the time-out.
__device__ __forceinline__ void kr_barrier(const KRArgs &A, bool cross, unsigned long long &epoch, unsigned &gen) {
    cross = cross && A.n_rank > 1;
    if (cross) epoch += 1;
    gen += 1;
    __syncthreads();
    if (threadIdx.x == 0 && !cross && (A.opts & KR_OPT_FAST_BARRIER)) {
        // one word: a release-add to arrive (nothing comes back), then acquire-poll the same count
        const unsigned target = gen * gridDim.x;
        unsigned seen;
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(A.bar_count) : "memory");
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(A.bar_count) : "memory");
        } while (seen < target);
    } else if (threadIdx.x == 0) {
        if (cross) __threadfence_system();
        else __threadfence();
        const unsigned arrived = atomicAdd(A.bar_count, 1u) + 1u;
        if (arrived == gen * gridDim.x) {
            if (cross) {
                // every CTA's system fence completed before it arrived, so this rank's peer stores have been
                // performed: relaxed flag stores and a relaxed spin are enough (a system-scope fence costs
                // microseconds, so there is exactly one per CTA per barrier)
                for (int g = 0; g < A.n_rank; ++g)
                    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(A.xflag[g] + A.rank), "l"(epoch) : "memory");
                const long long t0 = clock64();
                for (int g = 0; g < A.n_rank; ++g) {
                    const unsigned long long *mine = A.xflag[A.rank] + g;
                    unsigned long long seen;
                    do {
                        asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(mine) : "memory");
                        if (seen < epoch && clock64() - t0 > A.peer_timeout) {
                            for (int i = 0; i < P_COUNT; ++i)
                                A.part[(int64_t)i * A.n_chunks] = __longlong_as_double(0x7ff8000000000000LL);
                            A.timers->sync[T_FIX] = -1;
                            seen = epoch;
                        }
                    } while (seen < epoch);
                }
            }
            asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(A.bar_gen), "r"(gen) : "memory");
            __threadfence();                           // this CTA reads what the others (and the peers) wrote, too
        } else {
            unsigned g2;
            do {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(g2) : "l"(A.bar_gen) : "memory");
            } while (g2 < gen);
        }
        // what the peers wrote lies in this GPU's own memory: the gpu-scope acquire above (L1 invalidation) is
        // all a reader needs
    }
    __syncthreads();
}

#define KR_PHASE(id, cross, call)                                              \
    do {                                                                       \
        const long long t0_ = clock64();                                       \
        call;                                                                  \
        const long long t1_ = clock64();                                       \
        kr_barrier(A, cross, epoch, gen);                                      \
        if (id == T_SPMV && threadIdx.x == 0) *my_spmv += t1_ - t0_;           \
        if (timing) {                                                          \
            const long long t2_ = clock64();                                   \
            tim_work[id] += t1_ - t0_;                                         \
            tim_sync[id] += t2_ - t1_;                                         \
        }                                                                      \
    } while (0)
// a phase that may hand over through flagged partials: without the barrier the wait is inside the reduction that follows
#define KR_PHASE_B(id, barrier, call)                                          \
    do {                                                                       \
        const long long t0_ = clock64();                                       \
        call;                                                                  \
        const long long t1_ = clock64();                                       \
        if (barrier) kr_barrier(A, true, epoch, gen);                          \
        if (timing) {                                                          \
            const long long t2_ = clock64();                                   \
            tim_work[id] += t1_ - t0_;                                         \
            tim_sync[id] += t2_ - t1_;                                         \
        }                                                                      \
    } while (0)
// the reduction of the per-chunk partials every CTA repeats after a barrier (timed in the T_FIX slot)
#define KR_REDUCE(call)                                                        \
    do {                                                                       \
        const long long tr_ = clock64();                                       \
        call;                                                                  \
        if (timing) tim_work[T_FIX] += clock64() - tr_;                        \
    } while (0)
// a decision taken by thread 0 on the shared scalars, then published to the CTA
#define KR_SCALAR(which, r)                                                    \
    do {                                                                       \
        const long long ts_ = clock64();                                       \
        if (threadIdx.x == 0) scalar_step(S, which, r);                        \
        __syncthreads();                                                       \
        if (timing) tim_work[T_SCALAR] += clock64() - ts_;                     \
    } while (0)

template <bool SLAB, int CNT>
__global__ void __launch_bounds__(KR_THREADS, 1) k_kr_persistent(KRArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem sm = carve_smem(smem_raw);
    double *s_red = sm.red;
    KRScalars &S = *sm.ctl;
    if (threadIdx.x == 0) {
        S = *A.ctl;
        if (SLAB) mbar_init(sm.mbar, 1);
    }
    __syncthreads();
    const int nc = A.n_chunks;
    double *ybuf[2] = {A.y0, A.y1};
    const bool timing = (blockIdx.x == 0 && threadIdx.x == 0);
    const long long t_begin = clock64();
    unsigned long long epoch = A.n_rank > 1 ? *A.epoch : 0ull;
    unsigned gen = 0;
    long long *my_spmv = (long long *)(smem_raw + SM_STATE + 16);      // this CTA's own SpMV time (diagnostics)
    // CTA 0's phase timers live in shared memory while the loop runs (a global read-modify-write per phase
    // would sit on the critical path of every grid barrier)
    long long *tim_work = (long long *)(smem_raw + SM_TIM), *tim_sync = tim_work + T_COUNT;
    if (threadIdx.x == 0) {
        *my_spmv = 0;
        for (int i = 0; i < 2 * T_COUNT; ++i) tim_work[i] = 0;
    }

    // Hand-overs that carry only reduction partials can go through flagged words instead of a barrier: on one GPU all
    // three of them (KR_OPT_LL_PARTIALS, off: measured slower than the 1.5 us grid barrier); across GPUs the one after
    // `w` (KR_OPT_PEER_LL_W), where the alternative is a system-scope fence plus a flag round over the NVLink.
    const bool ll_single = A.n_rank <= 1 && (A.opts & KR_OPT_LL_PARTIALS);
    const bool ll_w = ll_single || (A.n_rank > 1 && (A.opts & KR_OPT_PEER_LL_W));
    unsigned ll_epoch = 0;

    int mode = -1;                                        // -1: first trip (x = 1)
    for (;;) {
        if (mode < 0) KR_PHASE(T_INIT, true, phase_init_p(A));
        else if (mode == KR_STATE_INNER) KR_PHASE(T_DIR, false, phase_dir_all(A, S.k == 1, S.beta, ybuf[S.ysel]));
        else KR_PHASE(T_UPDATE, true, phase_update<true>(A, S.ymode, S.gamma, S.alpha, ybuf[S.ysel]));
        const double *opnd = mode == KR_STATE_INNER ? A.u : A.x;                 // what the product is taken with ...
        const double *mult = CNT ? (mode == KR_STATE_INNER ? A.us : A.xs) : opnd;    // ... and what the stream multiplies
        KR_PHASE(T_SPMV, false, (phase_spmv<SLAB, CNT>(A, mult, sm)));
        if (mode == KR_STATE_INNER) {
            {
                double r[2];
                const int ids[2] = {PA, PB};
                const unsigned ll = ll_w ? ++ll_epoch : 0u;
                KR_PHASE_B(T_W, !ll_w, phase_w(A, s_red, ll));
                KR_REDUCE((reduce_parts<2, 0>(A, nc, ids, r, s_red, ll_w ? 1u : 0u, ll)));   // PB dates from the residual phase
                KR_SCALAR(KRS_ALPHA, r);
            }
            {
                double r[5];
                const int ids[5] = {PC, PMIN, PNEGMAX, PG1, PG2};
                const unsigned ll = ll_single ? ++ll_epoch : 0u;
                KR_PHASE_B(T_STEP, !ll_single,
                           phase_step(A, S.alpha, S.delta, S.Delta, ybuf[S.ysel], ybuf[S.ysel ^ 1], s_red, ll));
                KR_REDUCE((reduce_parts<1, 4>(A, nc, ids, r, s_red, ll_single ? 31u : 0u, ll)));
                KR_SCALAR(KRS_DECIDE, r);
            }
        } else {
            double r[1];
            const int ids[1] = {PA};
            const unsigned ll = ll_single ? ++ll_epoch : 0u;
            KR_PHASE_B(T_RESID, !ll_single, phase_resid(A, opnd, s_red, ll));
            KR_REDUCE((reduce_parts<1, 0>(A, nc, ids, r, s_red, ll_single ? 1u : 0u, ll)));
            KR_SCALAR(mode < 0 ? KRS_OUTER_FIRST : KRS_OUTER, r);
        }
        mode = S.state;
        if (mode == KR_STATE_DONE) break;
        __syncthreads();                                  // everybody has read the state before thread 0 moves on
    }
    // the scale vector leaves the exchange buffer before anybody can start another run on it
    if (A.xout != nullptr)
        for (int64_t r = (int64_t)blockIdx.x * KR_THREADS + threadIdx.x; r < A.n; r += (int64_t)gridDim.x * KR_THREADS)
            A.xout[r] = __ldcg(A.x + r);
    if (threadIdx.x == 0) A.cta_spmv[blockIdx.x] = *my_spmv;
    if (timing) {
        *A.ctl = S;
        for (int i = 0; i < T_COUNT; ++i) {
            A.timers->work[i] += tim_work[i];
            A.timers->sync[i] += tim_sync[i];
        }
        A.timers->total = clock64() - t_begin;
        if (A.n_rank > 1) *A.epoch = epoch;
    }
}

// ---- building the stream (once per balancing run) ---------------------------------------------------
// Columns are sorted within a row, so the entries of row r that fall in slab s are one contiguous
// segment.  Pass 1 (k_cell_bounds, a thread per cell) finds every cell's first entry by bisection and writes the
// padded segment length into cnt[s * npad + r]; the slab totals are padded to whole tiles; an exclusive scan gives
// the position vp of every cell; a second scan numbers the non-empty cells; pass 2 (k_stream_fill) copies the
// segments piece by piece.
// Every segment is padded with zero entries to a whole number of 8-entry pieces, so a segment can only start at
// the first entry of a lane's piece: the SpMV adds a piece up unconditionally and looks at ONE flag per piece.
__host__ __device__ __forceinline__ int64_t seg_padded(int64_t len) { return (len + SPMV_EPP - 1) & ~(int64_t)(SPMV_EPP - 1); }

// set the start flag of logical stream position `pos` (bit pos % 16 of the lane's 16-bit word)
__device__ __forceinline__ void stream_set_flag(uint16_t *sflag, int64_t pos) {
    const int64_t w16 = pos >> 4;                      // chunk * 32 + lane
    atomicOr((unsigned *)sflag + (w16 >> 1), (1u << (pos & 15)) << ((w16 & 1) * 16));
}

// Pass 1, one thread per (row, slab) cell: columns are sorted within a row, so the cell's entries are the run between
// two lower bounds.  cstart[v] = offset of the cell's first entry inside its row (k_cell_bounds, one bisection per
// cell); cnt[v] = its padded length, from the start of the same row's next cell (k_cell_len).
template <bool SLAB>
__global__ void __launch_bounds__(256) k_cell_bounds(KRArgs A, int32_t *__restrict__ cstart) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= A.nv) return;
    const int s = (int)(v / A.npad);
    const int64_t lr = v - (int64_t)s * A.npad;
    if (lr >= A.row_hi - A.row_lo || s == 0) {
        cstart[v] = 0;
        return;
    }
    const int64_t lo = A.indptr[lr], hi = A.indptr[lr + 1];
    const int32_t key = s * A.W;                       // first entry with column >= s * W, over the whole row: on an
    int64_t a = lo, b = hi;                            // unsorted row (which pass 2 reports) cells may then overlap or
    while (a < b) {                                    // come out of order, but never reach outside the row
        const int64_t mid = (a + b) >> 1;
        if (A.indices[mid] < key) a = mid + 1;
        else b = mid;
    }
    cstart[v] = (int32_t)(a - lo);
}

__global__ void __launch_bounds__(256) k_cell_len(KRArgs A, const int32_t *__restrict__ cstart, int64_t *__restrict__ cnt) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= A.nv) return;
    const int s = (int)(v / A.npad);
    const int64_t lr = v - (int64_t)s * A.npad;
    int64_t len = 0;
    if (lr < A.row_hi - A.row_lo) {
        const int64_t c0 = cstart[v];
        const int64_t c1 = s < A.S - 1 ? (int64_t)cstart[v + A.npad] : A.indptr[lr + 1] - A.indptr[lr];
        len = c1 > c0 ? c1 - c0 : 0;
    }
    cnt[v] = seg_padded(len);
}

// Pass 2: copy the cells into the stream.  A warp takes 32 consecutive cells (same slab, consecutive rows) and spreads
// their 8-entry PIECES over its four 8-lane groups -- a piece is eight consecutive CSR entries in and eight physically
// consecutive stream entries (one 32-byte sector of the packed form) out, so a long cell does not hold up a lane and a
// short one does not idle 31.  The last piece of a cell carries its zero padding; the first one sets the start flag.
// Entries are checked against their cell's column range: an unsorted or out-of-range row shows up here.
template <bool SLAB, bool SPREAD = false>
__global__ void __launch_bounds__(256) k_stream_fill(KRArgs A, const int32_t *__restrict__ cstart, double *__restrict__ sval,
                                                     void *__restrict__ scol_v, uint16_t *__restrict__ sflag) {
    const unsigned lane = lane_id(), grp = lane >> 3, sub = lane & 7u;
    const int64_t nw = (int64_t)gridDim.x * 8;
    const int n_local = A.row_hi - A.row_lo;
    const int64_t n_batch = A.nv >> 5;                 // npad is a multiple of 1024: whole batches, one slab each
    bool bad = false, bad16 = false;
    for (int64_t bt = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); bt < n_batch; bt += nw) {
        const int64_t v = bt * 32 + lane;
        const int s = (int)(v / A.npad);
        const int64_t lr = v - (int64_t)s * A.npad;
        int64_t c_src = 0, c_dst = 0;
        int c_len = 0;
        if (lr < n_local) {
            const int64_t lo = A.indptr[lr], hi = A.indptr[lr + 1];
            const int32_t c0 = cstart[v];
            const int64_t c1 = s < A.S - 1 ? (int64_t)cstart[v + A.npad] : hi - lo;
            c_src = lo + c0;
            c_len = c1 > c0 ? (int)(c1 - c0) : 0;
            bad |= c1 < c0;                            // boundaries out of order: the row is not sorted
            c_dst = A.vp[v];
        }
        const int np = (c_len + SPMV_EPP - 1) / SPMV_EPP;
        int off = np;                                  // inclusive scan over the lanes, then exclusive
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(kFullMask, off, d);
            if ((int)lane >= d) off += t;
        }
        const int total = __shfl_sync(kFullMask, off, 31);
        off -= np;
        const int col_lo = s * A.W, col_hi = (s == A.S - 1) ? A.n : (s + 1) * A.W;
        for (int t0 = 0; t0 < total; t0 += 4) {
            // which cell holds piece t0 + g: the highest lane whose first piece is <= it
            unsigned m_own = 0;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const unsigned m = __ballot_sync(kFullMask, off <= t0 + g);
                if ((int)grp == g) m_own = m;
            }
            const int t = t0 + (int)grp;
            const int sel = 31 - __clz(m_own);
            const int64_t src = __shfl_sync(kFullMask, c_src, sel);
            const int64_t dst = __shfl_sync(kFullMask, c_dst, sel);
            const int len = __shfl_sync(kFullMask, c_len, sel);
            const int p = t - __shfl_sync(kFullMask, off, sel);
            if (t >= total) continue;
            const int k = p * SPMV_EPP + (int)sub;
            const bool valid = k < len;
            const int64_t e = src + k;
            int col = valid ? A.indices[e] : col_lo;
            if (col < col_lo || col >= col_hi) {       // reported through ctl->status; clamped to stay in bounds
                bad = true;
                col = col_lo;
            }
            const unsigned lc = (unsigned)(col - col_lo);
            // Where inside its piece an entry goes is free (a piece is added up whole).  At step i of a piece the 32
            // lanes of the SpMV gather u[col] of their own pieces' i-th entries from shared memory, 16 fp64 bank pairs
            // per half-warp: consecutive lanes hold consecutive pieces of one row, whose columns run on (dense blocks)
            // or are spread evenly, so entry i of all of them falls on the same one or two bank pairs.  Order a piece by
            // bank pair (descending for odd lanes) and rotate it by half the lane number: the lanes then walk the bank
            // pairs out of step with each other.
            // (SPREAD is a template parameter: the default build of this kernel must not carry the ranking's registers)
            unsigned slot = sub;
            if (SLAB && SPREAD) {
                const unsigned gmask = 0xffu << (8 * grp);
                const unsigned key = ((lc & 15u) << 3) | sub;
                unsigned rank = 0;
#pragma unroll
                for (int j = 0; j < 8; ++j) rank += __shfl_sync(gmask, key, j, 8) < key ? 1u : 0u;
                const unsigned pl = (unsigned)(((dst + (int64_t)p * SPMV_EPP) & (SPMV_CHUNK - 1)) >> 4);   // its lane
                slot = (((pl & 1u) ? 7u - rank : rank) - (pl >> 1)) & 7u;
            }
            const int64_t ph = stream_phys(dst + (int64_t)p * SPMV_EPP) + slot;
            if (A.cnt_stream) {
                const uint32_t cnt_e = valid ? A.cnt32[e] : 0u;
                if (A.cnt_stream == 2) {
                    ((uint32_t *)sval)[ph] = (cnt_e << 16) | lc;            // low 16 bits of the count | column
                    if (cnt_e > 0xffffu && col != A.row_lo + (int)(bt * 32 - (int64_t)s * A.npad) + sel) {
                        // the high part of this off-diagonal count goes to the side list (sorted afterwards: k_big_build)
                        const unsigned long long q = atomicAdd((unsigned long long *)&A.ctl->n_big, 1ull);
                        if (q < (unsigned long long)BIG_CAP) A.big_e[q] = (long long)e;
                        else bad16 = true;
                    }
                } else {
                    ((uint32_t *)sval)[ph] = cnt_e;
                }
            } else if (A.cnt32) {
                const int row = A.row_lo + (int)(bt * 32 - (int64_t)s * A.npad) + sel;
                sval[ph] = valid ? site_scaled(A.cnt32[e], A.sites[row], __ldg(A.sites + col)) : 0.0;
            } else {
                sval[ph] = valid ? A.data[e] : 0.0;
            }
            if (A.cnt_stream != 2) {
                if (SLAB) ((uint16_t *)scol_v)[ph] = (uint16_t)lc;
                else ((uint32_t *)scol_v)[ph] = lc;
            }
            if (k == 0) stream_set_flag(sflag, dst);
        }
    }
    if (bad) A.ctl->status = B3C_ERR_ARG;              // unsorted or out-of-range columns
    if (bad16) A.ctl->ovf16 = 1;
}

// one CTA per slab: pad the slab's entry count to whole tiles (the padding belongs to its last cell)
__global__ void __launch_bounds__(1024) k_slab_pad(KRArgs A, int64_t *__restrict__ cnt) {
    __shared__ int64_t s_w[33];
    const int s = blockIdx.x;
    int64_t v = 0;
    const int64_t *row = cnt + (int64_t)s * A.npad;
    int64_t v1 = 0, v2 = 0, v3 = 0;                     // four independent loads in flight per thread
    int64_t i = threadIdx.x;
    for (; i + 3 * 1024 < A.npad; i += 4 * 1024) {
        v += row[i];
        v1 += row[i + 1024];
        v2 += row[i + 2 * 1024];
        v3 += row[i + 3 * 1024];
    }
    for (; i < A.npad; i += 1024) v += row[i];
    v += v1 + v2 + v3;
    int64_t tot;
    block_scan_excl<int64_t>(v, s_w, &tot);
    if (threadIdx.x == 0) {
        const int64_t pad = (SPMV_TILE - tot % SPMV_TILE) % SPMV_TILE;
        cnt[(int64_t)s * A.npad + A.npad - 1] += pad;
    }
}

// flag[v] = 1 if cell v has entries (a second scan numbers the segments)
__global__ void __launch_bounds__(256) k_cell_flags(int64_t nv, const int64_t *__restrict__ vp, int64_t *__restrict__ flag) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v < nv) flag[v] = vp[v + 1] > vp[v] ? 1 : 0;
}

// seg_of / seg_row from the numbering
__global__ void __launch_bounds__(256) k_cell_index(int64_t nv, const int64_t *__restrict__ vp,
                                                    const int64_t *__restrict__ ord, int32_t *__restrict__ seg_of,
                                                    int32_t *__restrict__ seg_row) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nv) return;
    if (vp[v + 1] > vp[v]) {
        seg_of[v] = (int32_t)ord[v];
        seg_row[ord[v]] = (int32_t)v;
    } else {
        seg_of[v] = -1;
    }
}

// first chunk of every slab; zero the last tile of every slab (its padding; the fill overwrites the real part);
// flag the first entry of the slab's last cell in case it consists of padding only
template <bool SLAB>
__global__ void __launch_bounds__(256) k_slab_finish(KRArgs A, double *__restrict__ sval, void *__restrict__ scol_v,
                                                     uint16_t *__restrict__ sflag, int32_t *__restrict__ slab_t0) {
    const int s = blockIdx.x;
    if (s == A.S) {
        if (threadIdx.x == 0) slab_t0[s] = (int32_t)(A.vp[A.nv] / SPMV_CHUNK);
        return;
    }
    const int64_t begin = A.vp[(int64_t)s * A.npad], end = A.vp[(int64_t)(s + 1) * A.npad];
    if (threadIdx.x == 0) slab_t0[s] = (int32_t)(begin / SPMV_CHUNK);
    const int64_t z0 = end - begin >= SPMV_TILE ? end - SPMV_TILE : begin;
    for (int64_t i = z0 + threadIdx.x; i < end; i += 256) {
        if (A.cnt_stream) ((uint32_t *)sval)[i] = 0u;
        else sval[i] = 0.0;
        if (SLAB) ((uint16_t *)scol_v)[i] = 0;
        else ((uint32_t *)scol_v)[i] = 0;
    }
    __syncthreads();
    const int64_t last = A.vp[(int64_t)(s + 1) * A.npad - 1];
    if (threadIdx.x == 0 && last < end) stream_set_flag(sflag, last);
}

// Bank order (slab form).  At step i of a chunk the 32 lanes of a warp gather u[col] for the i-th entry of their
// own 16-entry runs at once; u sits in shared memory as fp64, so an entry's bank pair is col % 16 and a
// half-warp whose 16 columns were drawn at random needs ~3 passes.  The order of the entries INSIDE a segment
// is free (the row sum is the only thing that depends on it, and it is fixed once per stream), so every lane
// orders each piece of a segment inside its run by (bank - lane) mod 16: lane l then tends to touch bank
// l + i at step i and the half-warp's banks are (nearly) distinct.  One thread per lane run, in place: the
// 16 entries of a run are touched by nobody else; flags belong to positions and do not move.
__global__ void __launch_bounds__(256) k_stream_bank_order(int64_t n_runs, double *__restrict__ sval,
                                                           uint16_t *__restrict__ scol, const uint16_t *__restrict__ sflag) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_runs) return;
    const int64_t chunk = t >> 5;
    const unsigned lane = (unsigned)(t & 31);
    const int64_t base = chunk * SPMV_CHUNK + SPMV_EPP * lane;          // piece 0; piece 1 is SPMV_CHUNK / 2 further
    double a[16];
    unsigned c[16];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const double4 *pv = (const double4 *)(sval + base + k * (SPMV_CHUNK / 2));
        const double4 v0 = pv[0], v1 = pv[1];
        a[8 * k + 0] = v0.x; a[8 * k + 1] = v0.y; a[8 * k + 2] = v0.z; a[8 * k + 3] = v0.w;
        a[8 * k + 4] = v1.x; a[8 * k + 5] = v1.y; a[8 * k + 6] = v1.z; a[8 * k + 7] = v1.w;
        const uint4 cc = *(const uint4 *)(scol + base + k * (SPMV_CHUNK / 2));
        c[8 * k + 0] = cc.x & 0xffffu; c[8 * k + 1] = cc.x >> 16; c[8 * k + 2] = cc.y & 0xffffu; c[8 * k + 3] = cc.y >> 16;
        c[8 * k + 4] = cc.z & 0xffffu; c[8 * k + 5] = cc.z >> 16; c[8 * k + 6] = cc.w & 0xffffu; c[8 * k + 7] = cc.w >> 16;
    }
    const unsigned fw = sflag[t];
    // sort key: pieces of different segments keep their order (segment ordinal inside the run), then the bank
    // rotated by the lane, then the position (a strict order, so the ranks are a permutation)
    unsigned key[16];
    unsigned seg = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        seg += (fw >> i) & 1u;
        key[i] = (seg << 8) | (((c[i] - lane) & 15u) << 4) | (unsigned)i;
    }
    bool moved = false;
    unsigned rank[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        unsigned r = 0;
#pragma unroll
        for (int j = 0; j < 16; ++j) r += key[j] < key[i] ? 1u : 0u;
        rank[i] = r;
        moved |= r != (unsigned)i;
    }
    if (!moved) return;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int64_t dst = base + (rank[i] >> 3) * (SPMV_CHUNK / 2) + (rank[i] & 7);
        sval[dst] = a[i];
        scol[dst] = (uint16_t)c[i];
    }
}

// chunk_seg0[c] = ordinal of the first segment that starts at or after entry c * 128
__global__ void __launch_bounds__(256) k_chunk_seg0(int64_t n_chunks, int64_t nv, const int64_t *__restrict__ vp,
                                                    const int64_t *__restrict__ ord, int32_t *__restrict__ chunk_seg0) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chunks) return;
    const int64_t pos = c * SPMV_CHUNK;
    int64_t lo = 0, hi = nv;                  // first cell in [0, nv] with vp[cell] >= pos
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (vp[mid] >= pos) hi = mid;
        else lo = mid + 1;
    }
    chunk_seg0[c] = (int32_t)ord[lo];
}

// dfix[r] = 1 where the diagonal entry of (global) row r is absent or zero (sparse_utils.py:110-115)
__global__ void __launch_bounds__(256) k_diag_fix(int32_t row_lo, int32_t row_hi, const int64_t *__restrict__ indptr,
                                                  const int32_t *__restrict__ indices, const double *__restrict__ data,
                                                  const uint32_t *__restrict__ cnt32, const int32_t *__restrict__ sites,
                                                  double *__restrict__ dfix, KRScalars *ctl, int packed,
                                                  const double *__restrict__ inv_s) {
    // One thread per row: the columns of a row are sorted (k_stream_fill rejects the matrix otherwise), so the
    // diagonal is found by bisection instead of walking the row.
    const int64_t lr = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool z = false;
    if (lr < row_hi - row_lo) {
        int64_t lo = indptr[lr];
        const int64_t end = indptr[lr + 1];
        int64_t hi = end;
        const int32_t gr = row_lo + (int32_t)lr;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (indices[mid] < gr) lo = mid + 1;
            else hi = mid;
        }
        double d = 0.0;           // duplicates of the diagonal would be summed by scipy's diagonal()
        double hi16 = 0.0;        // packed stream: what the 16-bit counts of the diagonal entries leave out
        for (int64_t e = lo; e < end && indices[e] == gr; ++e) {
            d += cnt32 ? site_scaled(cnt32[e], sites[gr], sites[gr]) : data[e];
            if (packed) hi16 += (double)(cnt32[e] & 0xffff0000u);
        }
        z = (d == 0.0);
        // rows_q adds dfix * operand_i: 1 for a zero diagonal (Q2); (high part of c_ii) / s_i^2 in the packed form
        double f = z ? 1.0 : 0.0;
        if (packed && hi16 != 0.0) f = __dmul_rn(__dmul_rn(hi16, inv_s[gr]), inv_s[gr]);
        dfix[gr] = f;
    }
    const unsigned nz = __popc(__ballot_sync(kFullMask, z));
    if (lane_id() == 0 && nz) atomicAdd((unsigned long long *)&ctl->zero_diag, (unsigned long long)nz);
}

// Side list of the packed count stream (one CTA): sort the CSR positions the count pass collected -- position order
// is (row, column) order, so every run adds a row's terms in the same order --, look up row, column and the high part
// of each count, and set the sign bit of dfix on the rows the list names (after k_diag_fix).
__global__ void __launch_bounds__(1024) k_big_build(KRArgs A) {
    __shared__ long long s_e[BIG_CAP];
    const int nb = A.n_big;
    int m = 1;
    while (m < nb) m <<= 1;
    for (int i = threadIdx.x; i < m; i += blockDim.x) s_e[i] = i < nb ? A.big_e[i] : 0x7fffffffffffffffLL;
    __syncthreads();
    for (int k = 2; k <= m; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < m; i += blockDim.x) {
                const int l = i ^ j;
                if (l > i) {
                    const long long a = s_e[i], b = s_e[l];
                    const bool up = (i & k) == 0;
                    if ((a > b) == up) {
                        s_e[i] = b;
                        s_e[l] = a;
                    }
                }
            }
            __syncthreads();
        }
    const int n_local = A.row_hi - A.row_lo;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) {
        const long long e = s_e[i];
        int lo = 0, hi = n_local;                      // last local row with indptr[row] <= e
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (A.indptr[mid] <= e) lo = mid;
            else hi = mid;
        }
        A.big_e[i] = e;
        A.big_row[i] = A.row_lo + lo;
        A.big_col[i] = A.indices[e];
        A.big_hi[i] = (double)(A.cnt32[e] & 0xffff0000u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nb; i += blockDim.x) {
        const int32_t r = A.big_row[i];
        if (i == 0 || A.big_row[i - 1] != r)
            A.dfix[r] = __longlong_as_double(__double_as_longlong(A.dfix[r]) | (long long)0x8000000000000000ULL);
    }
}

// ---- stand-alone kernels (microbench SpMV, host-driven phases, test hook) ----------------------------
// The multiplied vector is A.u: u itself for an fp64 stream (b3c_spmv, the phase API), or the staged u / s or x / s
// that b3c_kr_rowsum hands over in A.u for a counts stream (CNT 1 or 2, as k_kr_persistent).
template <bool SLAB, int CNT>
__global__ void __launch_bounds__(KR_THREADS, 1) k_spmv(KRArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem sm = carve_smem(smem_raw);
    if (SLAB) {
        if (threadIdx.x == 0) mbar_init(sm.mbar, 1);
        __syncthreads();
    }
    phase_spmv<SLAB, CNT>(A, A.u, sm);
}
// b3c_kr_rowsum: v staged as the KR phases stage their operand (put_x, phase_dir_all): opnd = v and, counts form,
// scaled = v * (1 / s) with the same rounding
__global__ void __launch_bounds__(256) k_kr_stage(int32_t n, const double *__restrict__ v, const double *__restrict__ inv_s,
                                                  double *__restrict__ opnd, double *__restrict__ scaled) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double x = v[i];
    opnd[i] = x;
    if (scaled) scaled[i] = __dmul_rn(x, __ldg(inv_s + i));
}
// b3c_kr_rowsum: the row sums of the local rows as phase_resid reads them (boundary_fix, then rows_q), one CTA per
// local chunk; q is indexed by local row
__global__ void __launch_bounds__(KR_THREADS) k_kr_rowsum(KRArgs A, const double *opnd, double *__restrict__ q) {
    const int c = A.row_lo / CHUNK + (int)blockIdx.x;
    double qq[CHUNK_RPT];
    boundary_fix(A, c);
    rows_q(A, opnd, c, qq);
#pragma unroll
    for (int i = 0; i < CHUNK_RPT; ++i) {
        const int64_t r = KR_ROW(c, i);
        if (r < A.row_hi) q[r - A.row_lo] = qq[i];
    }
}
// y[r] = (A u)[r] (b3c_spmv): one CTA per reduction chunk
__global__ void __launch_bounds__(KR_THREADS) k_spmv_collect(KRArgs A, double *__restrict__ y) {
    const int c = blockIdx.x;
    boundary_fix(A, c);
#pragma unroll
    for (int i = 0; i < CHUNK_RPT; ++i) {
        const int64_t r = KR_ROW(c, i);
        if (r >= A.row_lo && r < A.row_hi) y[r] = row_q(A, r);
    }
}

// ---- phase-at-a-time form (multi-GPU row-block driver) ------------------------------------------
// The driver all-reduces u with SUM, so the slices a rank does not own must hold zeros.
__device__ __forceinline__ void zero_nonlocal_u(const KRArgs &A) {
    if (A.row_lo == 0 && A.row_hi == A.n) return;
    KR_FOR_CHUNKS(c) {
        if (chunk_local(A, c)) continue;
#pragma unroll
        for (int i = 0; i < CHUNK_RPT; ++i) {
            const int64_t r = KR_ROW(c, i);
            if (r < A.n) A.u[r] = 0.0;
        }
    }
}

__global__ void __launch_bounds__(KR_THREADS) k_krp_phase(KRArgs A, int phase) {
    __shared__ double s_red[KR_WARPS * RED_MAX];
    const KRScalars S = *A.ctl;                 // only k_krp_scalar writes the control block
    double *ybuf[2] = {A.y0, A.y1};
    switch (phase) {
        case KRP_INIT:
            phase_init(A);
            zero_nonlocal_u(A);
            break;
        case KRP_RESID:
            phase_resid(A, A.u, s_red);
            break;
        case KRP_DIR:
            phase_dir(A, S.k == 1, S.beta, ybuf[S.ysel], s_red);
            zero_nonlocal_u(A);
            break;
        case KRP_W:
            phase_w(A, s_red);
            break;
        case KRP_STEP:
            phase_step(A, S.alpha, S.delta, S.Delta, ybuf[S.ysel], ybuf[S.ysel ^ 1], s_red);
            break;
        case KRP_UPDATE:
            phase_update<false>(A, S.ymode, S.gamma, S.alpha, ybuf[S.ysel]);
            zero_nonlocal_u(A);
            break;
        default:
            break;
    }
}

// the loop control of k_kr_persistent, one decision at a time, on the (all-reduced) partials
__global__ void __launch_bounds__(KR_THREADS) k_krp_scalar(KRArgs A, int which) {
    __shared__ double s_red[KR_WARPS * RED_MAX];
    KRScalars S = *A.ctl;
    const int nc = A.n_chunks;
    double r[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    if (which == KRS_OUTER_FIRST || which == KRS_OUTER) {
        double t[1];
        const int ids[1] = {PA};
        reduce_parts<1, 0>(A, nc, ids, t, s_red);
        r[0] = t[0];
    } else if (which == KRS_ALPHA) {
        double t[2];
        const int ids[2] = {PA, PB};
        reduce_parts<2, 0>(A, nc, ids, t, s_red);
        r[0] = t[0];
        r[1] = t[1];
    } else {
        const int ids[5] = {PC, PMIN, PNEGMAX, PG1, PG2};
        reduce_parts<1, 4>(A, nc, ids, r, s_red);
    }
    if (threadIdx.x == 0) {
        scalar_step(S, which, r);
        *A.ctl = S;
    }
}

static std::mutex g_krp_mu;
static std::unordered_map<void *, KRArgs> g_krp;

// ---- workspace ---------------------------------------------------------------------------------------
// tuning / test hooks (b3c_set_option): slab width cap and slab count cap of the SpMV operand
static std::atomic<int> g_slab_w_max{SLAB_W_MAX};
static std::atomic<int> g_slab_s_max{SLAB_S_MAX};
// KR_OPT_LL_PARTIALS stays off: measured slower than the barrier it replaces (profiles/r1_kr_phases.md)
// KR_OPT_BANK_ORDER stays off too: the reordering pass costs 91 us at C2 and saves 0.5 us per SpMV, so it would
// only pay for solves of more than ~180 SpMV (typical: 24-40)
// B3C_OPT_KR_COUNT_STREAM: the counts form streams uint32 counts (6 B per entry) instead of fp64 values (10 B)
static std::atomic<int> g_cnt_stream{2};
// KR_OPT_PIECE_SPREAD stays off as well: it takes 5 % of the u gather's shared-memory wavefronts away (C3: 592.8M -> 564.3M,
// KR kernel 5.11 -> 5.04 ms) but the ranking shuffles cost k_stream_fill more than that (0.60 -> 0.82 ms at C3, + 1.0 ms
// of set-up at C4 where the kernel gains nothing): profiles/raw/r4b_*, r4d_*, r4e_launch_table_c3_n1.md
static std::atomic<int> g_kr_opts{KR_OPT_SLAB_ALIGN | KR_OPT_FAST_BARRIER | KR_OPT_PEER_LL_W};
constexpr int BND_MAX = 148 * 2 + 8;                   // >= any SpMV grid

struct KRLayout {
    int32_t slab, S, W, n_chunks;
    int64_t nvec;                       // elements per (padded) vector
    int64_t nv_max, nnzv_max, nseg_max;
    int64_t o_dfix, o_inv_s, o_vec, o_qs, o_part, o_ll, o_ctl, o_timers, o_bar, o_bnd, o_cta;
    int64_t o_cnt, o_vp, o_ord, o_scan, o_slab_t0, o_sval, o_scol, o_sflag, o_seg0, o_seg_of, o_seg_row, o_big, o_cstart, total;
};

// `rows`: rows of the block the stream is built for (n for a whole matrix): the density rule counts the block's cells,
// and those are laid out for its rows padded to whole reduction chunks (npad, so nv = S * npad).  Counting the padded
// rows keeps a tail block of fewer than CHUNK rows in the form a CHUNK-row block with the same entries takes, which is
// what b3c_krp_workspace_bytes sizes for.
// `packed`: the stream will hold packed counts (b3c_kr_run*_counts with B3C_OPT_KR_COUNT_STREAM = 2)
static KRLayout kr_layout(int32_t n, int64_t nnz, int32_t rows, bool packed = false) {
    KRLayout L;
    Carver c;
    // Slab form whenever the matrix is at most B3C_OPT_KR_MAX_SLABS (16) slabs wide.  Wider matrices cut every row
    // into more (row, slab) segments, each padded to whole 8-entry pieces: that pays only while the segments are
    // long enough.  Measured on 1 M rows / 35 slabs (profiles/r1_spmv_sizes.md): 2.7 entries per cell -> gather
    // form 0.42 ms, slab form 0.69 ms; 9.2 per cell -> gather 1.37 ms, slab 1.06 ms; break-even near 5.
    const int64_t s_need = ceil_div(n, g_slab_w_max.load());
    const int s_max = g_slab_s_max.load();
    // (the packed count stream moves 4 B per padded entry against the gather form's 8 B plus an L1 wavefront per entry:
    // measured on C4's row blocks at 6 entries per cell, 1.9 us per million entries against 3.9)
    const int dense = packed ? SLAB_DENSE_CELL_PACKED : SLAB_DENSE_CELL;
    const bool dense_cells = s_max >= SLAB_S_MAX && s_need <= SLAB_S_CAP && nnz >= dense * align_up(rows, CHUNK) * s_need;
    L.slab = (s_need <= s_max || dense_cells) ? 1 : 0;
    L.S = L.slab ? (int32_t)s_need : 1;
    L.W = L.slab ? (int32_t)align_up(ceil_div(n, L.S), 2) : n;
    const int64_t npad_max = align_up(n, CHUNK);
    L.nv_max = (int64_t)L.S * npad_max;
    L.nseg_max = (nnz + L.S < L.nv_max ? nnz + L.S : L.nv_max) + 1;
    // every segment is padded to a whole piece (< SPMV_EPP extra entries each), every slab to a whole tile
    L.nnzv_max = align_up(nnz + (SPMV_EPP - 1) * L.nseg_max, SPMV_TILE) + (int64_t)L.S * SPMV_TILE;
    L.n_chunks = (int32_t)ceil_div(n, CHUNK);
    L.nvec = align_up(n, 32);
    L.o_dfix = c.take((int64_t)n * 8);
    L.o_inv_s = c.take(L.nvec * 8);
    L.o_vec = c.take(L.nvec * 8 * 11);
    L.o_qs = c.take(L.nseg_max * 8);
    L.o_part = c.take((int64_t)L.n_chunks * 8 * P_COUNT);
    L.o_ll = c.take((int64_t)L.n_chunks * 16 * P_COUNT + 128);       // + the arrival counter of the hand-overs
    L.o_ctl = c.take(sizeof(KRScalars));
    L.o_timers = c.take(sizeof(KRTimers));
    L.o_bar = c.take(256);
    L.o_bnd = c.take((int64_t)BND_MAX * (8 + 8 + 4 + 4 + 4));
    L.o_cta = c.take((int64_t)BND_MAX * 8);
    L.o_cnt = c.take((L.nv_max + 1) * 8);
    L.o_vp = c.take((L.nv_max + 1) * 8);
    L.o_ord = c.take((L.nv_max + 1) * 8);
    L.o_scan = c.take(scan_tmp_elems(L.nv_max) * 8);
    L.o_slab_t0 = c.take((SLAB_S_CAP + 2) * 4);
    L.o_sval = c.take(L.nnzv_max * 8);
    L.o_scol = c.take(L.nnzv_max * (L.slab ? 2 : 4));
    L.o_sflag = c.take(L.nnzv_max / 8 + 64);
    L.o_seg0 = c.take((L.nnzv_max / SPMV_CHUNK + 1) * 4);
    L.o_seg_of = c.take(L.nv_max * 4);
    L.o_seg_row = c.take(L.nseg_max * 4);
    L.o_big = c.take((int64_t)BIG_CAP * (8 + 4 + 4 + 8));
    L.o_cstart = c.take(L.nv_max * 4);
    L.total = c.cur;
    return L;
}

static void kr_bind(KRArgs &A, const KRLayout &L, char *ws, int32_t n, int32_t row_lo, int32_t row_hi, int64_t nnz,
                    const int64_t *indptr, const int32_t *indices, const double *data) {
    const int32_t n_local = row_hi - row_lo;
    A.n = n;
    A.row_lo = row_lo;
    A.row_hi = row_hi;
    A.nnz = nnz;
    A.indptr = indptr;
    A.indices = indices;
    A.data = data;
    A.cnt32 = nullptr;
    A.sites = nullptr;
    A.slab = L.slab;
    A.S = L.S;
    A.W = L.W;
    A.npad = (int32_t)align_up(n_local, CHUNK);
    A.nv = (int64_t)L.S * A.npad;
    A.nnzv = 0;                                        // known after the scan (kr_prepare)
    A.n_sch = 0;
    A.n_seg = 0;
    A.sval = (const double *)(ws + L.o_sval);
    A.scol = (const void *)(ws + L.o_scol);
    A.sflag = (const uint16_t *)(ws + L.o_sflag);
    A.chunk_seg0 = (const int32_t *)(ws + L.o_seg0);
    A.seg_of = (const int32_t *)(ws + L.o_seg_of);
    A.seg_row = (const int32_t *)(ws + L.o_seg_row);
    A.slab_c0 = (const int32_t *)(ws + L.o_slab_t0);
    A.qs = (double *)(ws + L.o_qs);
    A.n_bnd = 0;
    char *b = ws + L.o_bnd;
    A.bnd_head = (double *)b;
    A.bnd_tail = (double *)(b + (int64_t)BND_MAX * 8);
    A.bnd_flag = (int32_t *)(b + (int64_t)BND_MAX * 16);
    A.bnd_ord = (int32_t *)(b + (int64_t)BND_MAX * 20);
    A.bnd_lr = (int32_t *)(b + (int64_t)BND_MAX * 24);
    A.cnt = (int64_t *)(ws + L.o_cnt);
    A.vp = (int64_t *)(ws + L.o_vp);
    A.ord = (int64_t *)(ws + L.o_ord);
    A.scan_tmp = (int64_t *)(ws + L.o_scan);
    A.dfix = (double *)(ws + L.o_dfix);
    double *vec = (double *)(ws + L.o_vec);
    A.x = vec;
    A.v = vec + L.nvec * 1;
    A.rk = vec + L.nvec * 2;
    A.y0 = vec + L.nvec * 3;
    A.y1 = vec + L.nvec * 4;
    A.p = vec + L.nvec * 5;
    A.Z = vec + L.nvec * 6;
    A.w = vec + L.nvec * 7;
    A.u = vec + L.nvec * 8;
    A.us = vec + L.nvec * 9;
    A.xs = vec + L.nvec * 10;
    A.inv_s = (const double *)(ws + L.o_inv_s);
    A.cnt_stream = 0;
    A.n_big = 0;
    A.cstart = (int32_t *)(ws + L.o_cstart);
    A.big_e = (long long *)(ws + L.o_big);
    A.big_hi = (double *)(ws + L.o_big + (int64_t)BIG_CAP * 8);
    A.big_row = (int32_t *)(ws + L.o_big + (int64_t)BIG_CAP * 16);
    A.big_col = (int32_t *)(ws + L.o_big + (int64_t)BIG_CAP * 20);
    A.part = (double *)(ws + L.o_part);
    A.ll = (unsigned long long *)(ws + L.o_ll);
    A.n_chunks = L.n_chunks;
    A.ctl = (KRScalars *)(ws + L.o_ctl);
    A.timers = (KRTimers *)(ws + L.o_timers);
    A.bar_count = (unsigned *)(ws + L.o_bar);
    A.bar_gen = (unsigned *)(ws + L.o_bar + 128);
    A.opts = g_kr_opts.load();
    A.peer_timeout = g_peer_timeout_cycles.load();
    A.cta_spmv = (long long *)(ws + L.o_cta);
    A.n_rank = 0;
    A.rank = 0;
    A.epoch = nullptr;
    A.xout = nullptr;
    for (int g = 0; g < KR_MAX_RANKS; ++g) {
        A.xx[g] = nullptr;
        A.xz[g] = nullptr;
        A.xxs[g] = nullptr;
        A.xpart[g] = nullptr;
        A.xll[g] = nullptr;
        A.xflag[g] = nullptr;
    }
}

static unsigned row_warp_grid(int64_t n_rows) {
    int64_t blocks = ceil_div(n_rows > 0 ? n_rows : 1, 8);
    if (blocks > (int64_t)kNumSMs * 16) blocks = (int64_t)kNumSMs * 16;
    return (unsigned)blocks;
}

template <bool SLAB>
static int persistent_grid_of(int *grid_out) {
    static int cached = 0;
    if (!cached) {
        int per_sm = 0, per_sm_c = 0, dev = 0, sms = 0;
        const int smem = SLAB ? SM_BYTES_SLAB : SM_BYTES_GATHER;
        B3C_CUDA(cudaGetDevice(&dev));
        B3C_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        B3C_CUDA(cudaFuncSetAttribute(k_kr_persistent<SLAB, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        B3C_CUDA(cudaFuncSetAttribute(k_kr_persistent<SLAB, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        if (SLAB) B3C_CUDA(cudaFuncSetAttribute(k_kr_persistent<true, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        B3C_CUDA(cudaFuncSetAttribute(k_spmv<SLAB, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        B3C_CUDA(cudaFuncSetAttribute(k_spmv<SLAB, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        if (SLAB) B3C_CUDA(cudaFuncSetAttribute(k_spmv<true, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        B3C_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_kr_persistent<SLAB, 0>, KR_THREADS, smem));
        B3C_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_c, k_kr_persistent<SLAB, 1>, KR_THREADS, smem));
        if (per_sm < 1 || per_sm_c < 1) {
            set_error("persistent KR kernel does not fit on an SM");
            return B3C_ERR_CUDA;
        }
        cached = sms;                                  // one CTA per SM
        if (cached > BND_MAX) cached = BND_MAX;
    }
    *grid_out = cached;
    return B3C_OK;
}
static int persistent_grid(bool slab, int *grid_out) {
    return slab ? persistent_grid_of<true>(grid_out) : persistent_grid_of<false>(grid_out);
}

// inv_s[j] = 1 / s_j with zero site counts taken as one (contact_map.py:1103-1108, Q6)
__global__ void __launch_bounds__(256) k_inv_sites(int32_t n, const int32_t *__restrict__ sites, double *__restrict__ inv_s) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const int32_t sj = sites[i];
        inv_s[i] = __ddiv_rn(1.0, sj == 0 ? 1.0 : (double)sj);
    }
}

// Build the stream, its segment numbering and the zero-diagonal vector.  Needs the control block already
// uploaded (k_stream_fill / k_diag_fix write into it).  Two small D2H copies + syncs: the entry and segment counts
// size the fill; the fill reports bad columns and, in the packed form, how many large counts it met.
template <bool SLAB>
static int kr_prepare_t(KRArgs &A, const KRLayout &L, cudaStream_t s) {
    const int32_t n_local = A.row_hi - A.row_lo;
    double *sval = const_cast<double *>(A.sval);
    void *scol = const_cast<void *>(A.scol);
    uint16_t *sflag = const_cast<uint16_t *>(A.sflag);
    B3C_CUDA(cudaMemsetAsync(A.cnt + A.nv, 0, 8, s));
    B3C_CUDA(cudaMemsetAsync(sflag, 0, (size_t)(L.nnzv_max / 8 + 64), s));
    if (A.cnt_stream) {
        k_inv_sites<<<(unsigned)ceil_div(A.n, 256), 256, 0, s>>>(A.n, A.sites, const_cast<double *>(A.inv_s));
        B3C_LAUNCH_CHECK();
    }
    if (A.nv > 0) {
        k_cell_bounds<SLAB><<<(unsigned)ceil_div(A.nv, 256), 256, 0, s>>>(A, A.cstart);
        B3C_LAUNCH_CHECK();
        k_cell_len<<<(unsigned)ceil_div(A.nv, 256), 256, 0, s>>>(A, A.cstart, A.cnt);
        B3C_LAUNCH_CHECK();
    }
    k_slab_pad<<<(unsigned)A.S, 1024, 0, s>>>(A, A.cnt);
    B3C_LAUNCH_CHECK();
    int rc = scan_exclusive_i64(A.cnt, A.vp, A.nv, A.scan_tmp, s);
    if (rc) return rc;
    k_slab_finish<SLAB><<<(unsigned)A.S + 1, 256, 0, s>>>(A, sval, scol, sflag, const_cast<int32_t *>(A.slab_c0));
    B3C_LAUNCH_CHECK();
    // number the non-empty cells: cnt is reused for the 0/1 flags, ord receives their exclusive scan
    k_cell_flags<<<(unsigned)ceil_div(A.nv, 256), 256, 0, s>>>(A.nv, A.vp, A.cnt);
    B3C_LAUNCH_CHECK();
    rc = scan_exclusive_i64(A.cnt, A.ord, A.nv, A.scan_tmp, s);
    if (rc) return rc;
    int64_t totals[2] = {0, 0};
    KRScalars S;
    B3C_CUDA(cudaMemcpyAsync(&totals[0], A.vp + A.nv, 8, cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaMemcpyAsync(&totals[1], A.ord + A.nv, 8, cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaStreamSynchronize(s));
    if (totals[0] > L.nnzv_max || totals[0] % SPMV_TILE != 0 || totals[1] > L.nseg_max) {
        set_error("stream layout: %lld entries, %lld segments (capacity %lld, %lld)", (long long)totals[0],
                  (long long)totals[1], (long long)L.nnzv_max, (long long)L.nseg_max);
        return B3C_ERR_CAPACITY;
    }
    A.nnzv = totals[0];
    A.n_sch = A.nnzv / SPMV_CHUNK;
    A.n_seg = (int32_t)totals[1];
    const int64_t n_batch = A.nv / 32;
    const unsigned fill_grid = row_warp_grid(n_batch);                           // a warp per batch of 32 cells, grid-stride
    for (int attempt = 0; attempt < 2; ++attempt) {
        if (SLAB && (A.opts & KR_OPT_PIECE_SPREAD)) k_stream_fill<SLAB, true><<<fill_grid, 256, 0, s>>>(A, A.cstart, sval, scol, sflag);
        else k_stream_fill<SLAB><<<fill_grid, 256, 0, s>>>(A, A.cstart, sval, scol, sflag);
        B3C_LAUNCH_CHECK();
        B3C_CUDA(cudaMemcpyAsync(&S, A.ctl, sizeof(S), cudaMemcpyDeviceToHost, s));
        B3C_CUDA(cudaStreamSynchronize(s));
        if (S.status == B3C_ERR_ARG) {
            set_error("KR: column indices must be sorted within rows and lie in [0, n)");
            return B3C_ERR_ARG;
        }
        if (A.cnt_stream == 2 && S.ovf16) {            // more large off-diagonal counts than the side list holds:
            A.cnt_stream = 1;                          // fill again with 32-bit counts
            continue;
        }
        break;
    }
    A.n_big = A.cnt_stream == 2 ? (int32_t)S.n_big : 0;       // (at most BIG_CAP, or ovf16 would be set)
    if (SLAB && !A.cnt_stream && (A.opts & KR_OPT_BANK_ORDER) && A.n_sch > 0) {
        k_stream_bank_order<<<(unsigned)ceil_div(A.n_sch * 32, 256), 256, 0, s>>>(A.n_sch * 32, sval, (uint16_t *)scol, sflag);
        B3C_LAUNCH_CHECK();
    }
    k_cell_index<<<(unsigned)ceil_div(A.nv, 256), 256, 0, s>>>(A.nv, A.vp, A.ord, const_cast<int32_t *>(A.seg_of),
                                                               const_cast<int32_t *>(A.seg_row));
    B3C_LAUNCH_CHECK();
    const int64_t n_c = A.nnzv / SPMV_CHUNK;
    if (n_c > 0) {
        k_chunk_seg0<<<(unsigned)ceil_div(n_c, 256), 256, 0, s>>>(n_c, A.nv, A.vp, A.ord,
                                                                  const_cast<int32_t *>(A.chunk_seg0));
        B3C_LAUNCH_CHECK();
    }
    B3C_CUDA(cudaMemsetAsync(A.qs, 0, (size_t)(A.n_seg + 1) * 8, s));
    k_diag_fix<<<(unsigned)ceil_div(n_local > 0 ? n_local : 1, 256), 256, 0, s>>>(A.row_lo, A.row_hi, A.indptr, A.indices, A.data, A.cnt32, A.sites,
                                                              A.dfix, A.ctl, A.cnt_stream == 2 ? 1 : 0, A.inv_s);
    B3C_LAUNCH_CHECK();
    if (A.n_big > 0) {
        k_big_build<<<1, 1024, 0, s>>>(A);
        B3C_LAUNCH_CHECK();
    }
    rc = persistent_grid(SLAB, &A.n_bnd);
    return rc;
}
static int kr_prepare(KRArgs &A, const KRLayout &L, cudaStream_t s) {
    return A.slab ? kr_prepare_t<true>(A, L, s) : kr_prepare_t<false>(A, L, s);
}

// the stand-alone SpMV of the stream's form; A.u is the vector it multiplies (see k_spmv)
static int launch_spmv(const KRArgs &A, cudaStream_t s) {
    if (A.slab) {
        if (A.cnt_stream == 2) k_spmv<true, 2><<<A.n_bnd, KR_THREADS, SM_BYTES_SLAB, s>>>(A);
        else if (A.cnt_stream) k_spmv<true, 1><<<A.n_bnd, KR_THREADS, SM_BYTES_SLAB, s>>>(A);
        else k_spmv<true, 0><<<A.n_bnd, KR_THREADS, SM_BYTES_SLAB, s>>>(A);
    } else {
        if (A.cnt_stream) k_spmv<false, 1><<<A.n_bnd, KR_THREADS, SM_BYTES_GATHER, s>>>(A);
        else k_spmv<false, 0><<<A.n_bnd, KR_THREADS, SM_BYTES_GATHER, s>>>(A);
    }
    B3C_LAUNCH_CHECK();
    return B3C_OK;
}

static void kr_scalars_init(KRScalars &S, double tol, double delta, double Delta, int32_t max_iter) {
    memset(&S, 0, sizeof(S));
    S.tol = tol;
    S.delta = delta;
    S.Delta = Delta;
    S.rt = tol * tol;                 // sparse_utils.py:135
    S.stop_tol = tol * 0.5;           // sparse_utils.py:131
    S.eta = 0.1;                      // etamax (sparse_utils.py:129-130)
    S.max_iter = max_iter;
}

}  // namespace b3c

using namespace b3c;

extern "C" {

int b3c_set_option(int32_t key, int64_t value) {
    switch (key) {
        case B3C_OPT_KR_SLAB_WIDTH:
            B3C_REQUIRE(value >= 2 && value <= SLAB_W_MAX, "slab width must be in [2, %d]", SLAB_W_MAX);
            g_slab_w_max.store((int)value & ~1);
            return B3C_OK;
        case B3C_OPT_KR_MAX_SLABS:
            B3C_REQUIRE(value >= 0 && value <= SLAB_S_CAP, "slab count cap must be in [0, %d]", SLAB_S_CAP);
            g_slab_s_max.store((int)value);
            return B3C_OK;
        case B3C_OPT_KR_FLAGS:
            B3C_REQUIRE(value >= 0 && value <= 255, "KR option flags must be in [0, 255]");
            g_kr_opts.store((int)value);
            return B3C_OK;
        case B3C_OPT_KR_COUNT_STREAM:
            B3C_REQUIRE(value >= 0 && value <= 2, "count stream option is 0, 1 or 2");
            g_cnt_stream.store((int)value);
            return B3C_OK;
        case B3C_OPT_USE_GRAPHS:
            B3C_REQUIRE(value == 0 || value == 1, "graph option is 0 or 1");
            g_use_graphs.store((int)value);
            return B3C_OK;
        case B3C_OPT_PEER_TIMEOUT_MS:
            B3C_REQUIRE(value >= 1 && value <= 3600000, "peer time-out must be between 1 ms and one hour");
            g_peer_timeout_cycles.store((long long)value * 2000000LL);        // SM cycles at ~2 GHz
            return B3C_OK;
        default:
            set_error("unknown option %d", key);
            return B3C_ERR_ARG;
    }
}

int64_t b3c_kr_workspace_bytes(int32_t n, int64_t nnz) {
    if (n <= 0 || nnz < 0) return B3C_ERR_ARG;
    // the fp64 and the packed-count form of one matrix may choose differently between slab and gather: room for either
    const int64_t a = kr_layout(n, nnz, n, false).total, b = kr_layout(n, nnz, n, true).total;
    return a > b ? a : b;
}

// launch the persistent kernel on a prepared operand, wait, and report
static int kr_launch_collect(KRArgs &A, int32_t max_iter, double *d_x, int64_t *h_info, cudaStream_t s) {
    static thread_local cudaEvent_t ev[2] = {nullptr, nullptr};
    if (!ev[0]) {
        B3C_CUDA(cudaEventCreate(&ev[0]));
        B3C_CUDA(cudaEventCreate(&ev[1]));
    }
    const int grid = A.n_bnd;
    A.xout = d_x;                                       // the kernel leaves the whole scale vector here
    void *args[] = {&A};
    B3C_CUDA(cudaMemsetAsync(A.bar_count, 0, 256, s));
    B3C_CUDA(cudaMemsetAsync(A.ll, 0, (size_t)A.n_chunks * 16 * P_COUNT + 128, s));      // epoch 0 = never written
    B3C_CUDA(cudaEventRecord(ev[0], s));
    void *kern = A.slab ? (A.cnt_stream == 2 ? (void *)k_kr_persistent<true, 2>
                                             : A.cnt_stream ? (void *)k_kr_persistent<true, 1> : (void *)k_kr_persistent<true, 0>)
                        : (A.cnt_stream ? (void *)k_kr_persistent<false, 1> : (void *)k_kr_persistent<false, 0>);
    B3C_CUDA(cudaLaunchCooperativeKernel(kern, dim3(grid), dim3(KR_THREADS), args,
                                         A.slab ? SM_BYTES_SLAB : SM_BYTES_GATHER, s));
    B3C_CUDA(cudaEventRecord(ev[1], s));
    count_launch();
    KRScalars S;
    KRTimers T;
    long long cta[BND_MAX];
    B3C_CUDA(cudaMemcpyAsync(&S, A.ctl, sizeof(S), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaMemcpyAsync(&T, A.timers, sizeof(T), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaMemcpyAsync(cta, A.cta_spmv, (size_t)grid * 8, cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaStreamSynchronize(s));                // the one host synchronisation of the solve's result
    float ms = 0.f;
    B3C_CUDA(cudaEventElapsedTime(&ms, ev[0], ev[1]));
    h_info[0] = S.n_iter;
    h_info[1] = S.zero_diag;
    h_info[2] = S.outer;
    h_info[3] = S.n_spmv;
    h_info[4] = grid;
    h_info[5] = T.total;
    for (int i = 0; i < T_COUNT; ++i) {
        h_info[6 + i] = T.work[i];
        h_info[6 + T_COUNT + i] = T.sync[i];
    }
    h_info[24] = A.slab ? A.S : 0;
    h_info[25] = A.nnzv;
    h_info[26] = A.n_seg;
    h_info[31] = A.cnt_stream == 2 ? 4 : A.cnt_stream ? (A.slab ? 6 : 8) : (A.slab ? 10 : 12);      // stream bytes per entry
    h_info[27] = (int64_t)(ms * 1000.0f + 0.5f);       // the persistent kernel alone, microseconds (CUDA events)
    {
        long long mn = cta[0], mx = cta[0], sum = 0;
        for (int i = 0; i < grid; ++i) {
            mn = cta[i] < mn ? cta[i] : mn;
            mx = cta[i] > mx ? cta[i] : mx;
            sum += cta[i];
        }
        h_info[28] = mn;                               // SpMV cycles of the fastest / slowest CTA and the mean
        h_info[29] = mx;
        h_info[30] = sum / grid;
    }
    if (T.sync[T_FIX] < 0) {
        set_error("KR: a rank did not reach a cross-GPU barrier within the time-out");
        return B3C_ERR_CUDA;
    }
    if (S.status == B3C_ERR_TIE) {
        set_error("KR: max(ynew) == Delta with no element above Delta (reference raises ValueError here)");
        return B3C_ERR_TIE;
    }
    if (S.status == B3C_ERR_NAN) {
        set_error("scale vector has developed invalid values (NANs)!");
        return B3C_ERR_NAN;
    }
    if (S.status == B3C_ERR_NOCONV || S.n_iter > max_iter) {
        set_error("matrix balancing failed to converge in %lld iterations", (long long)S.n_iter);
        return B3C_ERR_NOCONV;
    }
    return B3C_OK;
}

// The stream form a counts matrix asks for under the current options (before the build's fall-back from 2 to 1)
static int32_t kr_cnt_stream(bool counts, bool slab) {
    const int cs = g_cnt_stream.load();
    return (counts && cs) ? ((cs == 2 && slab) ? 2 : 1) : 0;
}

// The SpMV operand of rows [row_lo, row_hi) as every KR entry point builds it: layout (the density rule over the
// block's rows), binding, the count-stream form, the control block, the stream with its side list and dfix.
// kr_run_impl, kr_run_peer_impl and b3c_kr_rowsum all go through here, so what the test hook sums is the product's
// operand.
static int kr_operand(KRArgs &A, KRLayout &L, int32_t n, int32_t row_lo, int32_t row_hi, int64_t nnz,
                      const int64_t *d_indptr, const int32_t *d_indices, const double *d_data, const uint32_t *d_counts,
                      const int32_t *d_sites, double tol, double delta, double Delta, int32_t max_iter, void *d_ws,
                      int64_t ws_bytes, cudaStream_t s) {
    L = kr_layout(n, nnz, row_hi - row_lo, !d_data && d_counts && g_cnt_stream.load() == 2);
    if (ws_bytes < L.total) {
        set_error("KR workspace too small: %lld < %lld", (long long)ws_bytes, (long long)L.total);
        return B3C_ERR_CAPACITY;
    }
    kr_bind(A, L, (char *)d_ws, n, row_lo, row_hi, nnz, d_indptr, d_indices, d_data);
    A.cnt32 = d_data ? nullptr : d_counts;
    A.sites = d_data ? nullptr : d_sites;
    A.cnt_stream = kr_cnt_stream(A.cnt32 != nullptr, A.slab);
    KRScalars S;
    kr_scalars_init(S, tol, delta, Delta, max_iter);
    B3C_CUDA(cudaMemcpyAsync(A.ctl, &S, sizeof(S), cudaMemcpyHostToDevice, s));
    B3C_CUDA(cudaMemsetAsync(A.timers, 0, sizeof(KRTimers), s));
    return kr_prepare(A, L, s);
}

static int kr_run_impl(int32_t n, int64_t nnz, const int64_t *d_indptr, const int32_t *d_indices, const double *d_data,
                       const uint32_t *d_counts, const int32_t *d_sites, double tol, double delta, double Delta,
                       int32_t max_iter, double *d_x, void *d_ws, int64_t ws_bytes, int64_t *h_info, void *stream) {
    B3C_REQUIRE(n > 0 && nnz >= 0 && d_indptr && d_x && d_ws && h_info, "bad arguments");
    B3C_REQUIRE(nnz == 0 || (d_indices && (d_data || (d_counts && d_sites))), "null matrix arrays");
    cudaStream_t s = (cudaStream_t)stream;
    KRArgs A;
    KRLayout L;
    int rc = kr_operand(A, L, n, 0, n, nnz, d_indptr, d_indices, d_data, d_counts, d_sites, tol, delta, Delta, max_iter,
                        d_ws, ws_bytes, s);
    if (rc) return rc;
    return kr_launch_collect(A, max_iter, d_x, h_info, s);
}

int b3c_kr_run(int32_t n, int64_t nnz, const int64_t *d_indptr, const int32_t *d_indices, const double *d_data,
               double tol, double delta, double Delta, int32_t max_iter, int32_t mode, double *d_x, void *d_ws,
               int64_t ws_bytes, int64_t *h_info, void *stream) {
    B3C_REQUIRE(mode == 0, "b3c_kr_run: only mode 0 (persistent kernel) is implemented; use b3c_krp_* for phases");
    B3C_REQUIRE(nnz == 0 || d_data, "null matrix values");
    return kr_run_impl(n, nnz, d_indptr, d_indices, d_data, nullptr, nullptr, tol, delta, Delta, max_iter, d_x, d_ws,
                       ws_bytes, h_info, stream);
}

int b3c_kr_run_counts(int32_t n, int64_t nnz, const int64_t *d_indptr, const int32_t *d_indices,
                      const uint32_t *d_counts, const int32_t *d_sites, double tol, double delta, double Delta,
                      int32_t max_iter, double *d_x, void *d_ws, int64_t ws_bytes, int64_t *h_info, void *stream) {
    B3C_REQUIRE(d_sites && (nnz == 0 || d_counts), "null counts / sites");
    return kr_run_impl(n, nnz, d_indptr, d_indices, nullptr, d_counts, d_sites, tol, delta, Delta, max_iter, d_x, d_ws,
                       ws_bytes, h_info, stream);
}

// ---- peer mode: one persistent kernel per GPU of a node, exchange buffers mapped over NVLink ------------
// exchange buffer of a rank: [flags: KR_MAX_RANKS x u64][epoch u64][x: nvec x f64][Z: nvec x f64][partials]
// [flagged partial words + their arrival counter]
struct XLayout {
    int64_t o_flag, o_epoch, o_x, o_xs, o_z, o_part, o_ll, total;
};
static XLayout x_layout(int32_t n) {
    XLayout X;
    Carver c;
    X.o_flag = c.take(KR_MAX_RANKS * 8);
    X.o_epoch = c.take(8);
    X.o_x = c.take(align_up(n, 32) * 8);
    X.o_xs = c.take(align_up(n, 32) * 8);
    X.o_z = c.take(align_up(n, 32) * 8);
    X.o_part = c.take(ceil_div(n, CHUNK) * 8 * P_COUNT);
    X.o_ll = c.take(ceil_div(n, CHUNK) * 16 * P_COUNT + 128);
    X.total = c.cur;
    return X;
}

int64_t b3c_kr_exchange_bytes(int32_t n) {
    if (n <= 0) return B3C_ERR_ARG;
    return x_layout(n).total;
}

int b3c_peer_alloc(int64_t bytes, void **d_ptr, uint8_t *h_handle) {
    B3C_REQUIRE(bytes > 0 && d_ptr && h_handle, "bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    void *p = nullptr;
    B3C_CUDA(cudaMalloc(&p, (size_t)bytes));
    B3C_CUDA(cudaMemset(p, 0, (size_t)bytes));
    cudaIpcMemHandle_t h;
    B3C_CUDA(cudaIpcGetMemHandle(&h, p));
    memcpy(h_handle, &h, sizeof(h));
    *d_ptr = p;
    return B3C_OK;
}
int b3c_peer_open(const uint8_t *h_handle, void **d_ptr) {
    B3C_REQUIRE(h_handle && d_ptr, "bad arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, h_handle, sizeof(h));
    B3C_CUDA(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return B3C_OK;
}
int b3c_peer_close(void *d_ptr) {
    B3C_CUDA(cudaIpcCloseMemHandle(d_ptr));
    return B3C_OK;
}
int b3c_peer_free(void *d_ptr) {
    B3C_CUDA(cudaFree(d_ptr));
    return B3C_OK;
}

static int kr_run_peer_impl(int32_t n, int32_t row_lo, int32_t row_hi, int64_t nnz_local, const int64_t *d_indptr,
                            const int32_t *d_indices, const double *d_data, const uint32_t *d_counts,
                            const int32_t *d_sites, double tol, double delta, double Delta, int32_t max_iter,
                            int32_t rank, int32_t n_ranks, void *const *h_exchange, double *d_x, void *d_ws,
                            int64_t ws_bytes, int64_t *h_info, void *stream) {
    B3C_REQUIRE(n > 0 && 0 <= row_lo && row_lo < row_hi && row_hi <= n, "bad row block [%d,%d) of %d", row_lo, row_hi, n);
    B3C_REQUIRE(row_lo % CHUNK == 0 && (row_hi % CHUNK == 0 || row_hi == n), "row blocks must be %d-row aligned", CHUNK);
    B3C_REQUIRE(d_indptr && d_x && d_ws && h_info && h_exchange && nnz_local >= 0, "bad arguments");
    B3C_REQUIRE(n_ranks >= 1 && n_ranks <= KR_MAX_RANKS && rank >= 0 && rank < n_ranks, "bad rank %d of %d (at most %d)",
                rank, n_ranks, KR_MAX_RANKS);
    for (int g = 0; g < n_ranks; ++g) B3C_REQUIRE(h_exchange[g] != nullptr, "null exchange buffer of rank %d", g);
    cudaStream_t s = (cudaStream_t)stream;
    KRArgs A;
    KRLayout L;
    int rc = kr_operand(A, L, n, row_lo, row_hi, nnz_local, d_indptr, d_indices, d_data, d_counts, d_sites, tol, delta,
                        Delta, max_iter, d_ws, ws_bytes, s);
    if (rc) return rc;
    const XLayout X = x_layout(n);
    for (int g = 0; g < n_ranks; ++g) {
        char *b = (char *)h_exchange[g];
        A.xflag[g] = (unsigned long long *)(b + X.o_flag);
        A.xx[g] = (double *)(b + X.o_x);
        A.xz[g] = (double *)(b + X.o_z);
        A.xxs[g] = (double *)(b + X.o_xs);
        A.xpart[g] = (double *)(b + X.o_part);
        A.xll[g] = (unsigned long long *)(b + X.o_ll);
    }
    A.n_rank = n_ranks;
    A.rank = rank;
    A.epoch = (unsigned long long *)((char *)h_exchange[rank] + X.o_epoch);
    // x, Z, the partials and their flagged words live in the exchange buffer: every rank's slice is written by its owner
    A.x = A.xx[rank];
    A.xs = A.xxs[rank];
    A.Z = A.xz[rank];
    A.part = A.xpart[rank];
    A.ll = A.xll[rank];
    return kr_launch_collect(A, max_iter, d_x, h_info, s);
}

int b3c_kr_run_peer(int32_t n, int32_t row_lo, int32_t row_hi, int64_t nnz_local, const int64_t *d_indptr,
                    const int32_t *d_indices, const double *d_data, double tol, double delta, double Delta,
                    int32_t max_iter, int32_t rank, int32_t n_ranks, void *const *h_exchange, double *d_x, void *d_ws,
                    int64_t ws_bytes, int64_t *h_info, void *stream) {
    B3C_REQUIRE(nnz_local == 0 || d_data, "null matrix values");
    return kr_run_peer_impl(n, row_lo, row_hi, nnz_local, d_indptr, d_indices, d_data, nullptr, nullptr, tol, delta, Delta,
                            max_iter, rank, n_ranks, h_exchange, d_x, d_ws, ws_bytes, h_info, stream);
}

int b3c_kr_run_peer_counts(int32_t n, int32_t row_lo, int32_t row_hi, int64_t nnz_local, const int64_t *d_indptr,
                           const int32_t *d_indices, const uint32_t *d_counts, const int32_t *d_sites, double tol,
                           double delta, double Delta, int32_t max_iter, int32_t rank, int32_t n_ranks,
                           void *const *h_exchange, double *d_x, void *d_ws, int64_t ws_bytes, int64_t *h_info,
                           void *stream) {
    B3C_REQUIRE(d_sites && (nnz_local == 0 || d_counts), "null counts / sites");
    return kr_run_peer_impl(n, row_lo, row_hi, nnz_local, d_indptr, d_indices, nullptr, d_counts, d_sites, tol, delta,
                            Delta, max_iter, rank, n_ranks, h_exchange, d_x, d_ws, ws_bytes, h_info, stream);
}

int b3c_spmv(int32_t n, int64_t nnz, const int64_t *d_indptr, const int32_t *d_indices, const double *d_data,
             const double *d_u, double *d_y, void *d_ws, int64_t ws_bytes, int32_t prepared, void *stream) {
    B3C_REQUIRE(n > 0 && nnz >= 0 && d_indptr && d_u && d_y && d_ws, "bad arguments");
    const KRLayout L = kr_layout(n, nnz, n);
    if (ws_bytes < L.total) {
        set_error("SpMV workspace too small: %lld < %lld", (long long)ws_bytes, (long long)L.total);
        return B3C_ERR_CAPACITY;
    }
    cudaStream_t s = (cudaStream_t)stream;
    KRArgs A;
    if (prepared) {
        std::lock_guard<std::mutex> g(g_krp_mu);
        auto it = g_krp.find(d_ws);
        B3C_REQUIRE(it != g_krp.end(), "b3c_spmv: workspace %p was not prepared", d_ws);
        A = it->second;
        B3C_REQUIRE(A.n == n && A.nnz == nnz && A.indptr == d_indptr, "b3c_spmv: workspace prepared for another matrix");
    } else {
        kr_bind(A, L, (char *)d_ws, n, 0, n, nnz, d_indptr, d_indices, d_data);
        B3C_CUDA(cudaMemsetAsync(A.ctl, 0, sizeof(KRScalars), s));
        int rc = kr_prepare(A, L, s);
        if (rc) return rc;
        std::lock_guard<std::mutex> g(g_krp_mu);
        g_krp[d_ws] = A;
    }
    if (A.slab) {
        // the TMA copy of a slab needs a 16-byte aligned, padded operand: stage it in the workspace
        B3C_CUDA(cudaMemcpyAsync(A.u, d_u, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
    } else {
        A.u = const_cast<double *>(d_u);
    }
    int rc = launch_spmv(A, s);
    if (rc) return rc;
    k_spmv_collect<<<(unsigned)A.n_chunks, KR_THREADS, 0, s>>>(A, d_y);
    B3C_LAUNCH_CHECK();
    return B3C_OK;
}

// ---- test hooks: the operand's layout and its row sums ------------------------------------------------
int b3c_kr_plan(int32_t n, int64_t nnz_local, int32_t rows, int32_t counts, int64_t *h_out) {
    B3C_REQUIRE(h_out != nullptr && n > 0 && nnz_local >= 0 && rows >= 1 && rows <= n, "bad arguments");
    const KRLayout L = kr_layout(n, nnz_local, rows, counts && g_cnt_stream.load() == 2);
    h_out[0] = L.slab ? L.S : 0;
    h_out[1] = L.S;
    h_out[2] = L.W;
    h_out[3] = kr_cnt_stream(counts != 0, L.slab != 0);
    h_out[4] = L.total;
    return B3C_OK;
}

int b3c_kr_rowsum(int32_t n, int32_t row_lo, int32_t row_hi, int64_t nnz_local, const int64_t *d_indptr,
                  const int32_t *d_indices, const double *d_data, const uint32_t *d_counts, const int32_t *d_sites,
                  int32_t which, const double *d_v, double *d_q, void *d_ws, int64_t ws_bytes, int64_t *h_info,
                  void *stream) {
    B3C_REQUIRE(n > 0 && 0 <= row_lo && row_lo < row_hi && row_hi <= n, "bad row block [%d,%d) of %d", row_lo, row_hi, n);
    B3C_REQUIRE(row_lo % CHUNK == 0 && (row_hi % CHUNK == 0 || row_hi == n), "row blocks must be %d-row aligned", CHUNK);
    B3C_REQUIRE(d_indptr && d_v && d_q && d_ws && h_info && nnz_local >= 0 && (which == 0 || which == 1), "bad arguments");
    B3C_REQUIRE(!d_data != !d_sites && (d_data || d_counts), "pass the values, or the counts and the sites");
    B3C_REQUIRE(nnz_local == 0 || d_indices, "null matrix arrays");
    cudaStream_t s = (cudaStream_t)stream;
    KRArgs A;
    KRLayout L;
    int rc = kr_operand(A, L, n, row_lo, row_hi, nnz_local, d_indptr, d_indices, d_data, d_counts, d_sites, 1e-6, 0.1,
                        3.0, 1000, d_ws, ws_bytes, s);
    if (rc) return rc;
    // v goes where the iteration keeps the operand it multiplies: u of a CG step (which = 0) or x of a residual
    // (which = 1); the other pair is filled with NaN so that a row sum reading the wrong one cannot pass
    double *opnd = which ? A.x : A.u, *scaled = which ? A.xs : A.us;
    B3C_CUDA(cudaMemsetAsync(which ? A.u : A.x, 0xff, (size_t)L.nvec * 8, s));
    B3C_CUDA(cudaMemsetAsync(which ? A.us : A.xs, 0xff, (size_t)L.nvec * 8, s));
    k_kr_stage<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(n, d_v, A.inv_s, opnd, A.cnt_stream ? scaled : nullptr);
    B3C_LAUNCH_CHECK();
    KRArgs B = A;
    B.u = A.cnt_stream ? scaled : opnd;
    rc = launch_spmv(B, s);
    if (rc) return rc;
    k_kr_rowsum<<<(unsigned)ceil_div(row_hi - row_lo, CHUNK), KR_THREADS, 0, s>>>(A, opnd, d_q);
    B3C_LAUNCH_CHECK();
    KRScalars S;
    B3C_CUDA(cudaMemcpyAsync(&S, A.ctl, sizeof(S), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaStreamSynchronize(s));
    h_info[0] = A.slab ? A.S : 0;
    h_info[1] = A.S;
    h_info[2] = A.cnt_stream == 2 ? 4 : A.cnt_stream ? (A.slab ? 6 : 8) : (A.slab ? 10 : 12);
    h_info[3] = A.n_big;
    h_info[4] = A.nnzv;
    h_info[5] = A.n_seg;
    h_info[6] = S.zero_diag;
    h_info[7] = L.total;
    return B3C_OK;
}

// ---- phase API (multi-GPU row-block driver, bin3c_b200/dist.py) --------------------------------------

int64_t b3c_krp_workspace_bytes(int32_t n, int64_t nnz_local) {
    if (n <= 0 || nnz_local < 0) return B3C_ERR_ARG;
    // the form (slab or gather) depends on how dense the block's cells are, i.e. on its row count, which is not known
    // here: room for either
    const int64_t a = kr_layout(n, nnz_local, n).total, b = kr_layout(n, nnz_local, CHUNK, true).total;
    return a > b ? a : b;
}

int b3c_krp_setup(int32_t n, int32_t row_lo, int32_t row_hi, int64_t nnz_local, const int64_t *d_indptr,
                  const int32_t *d_indices, const double *d_data, double tol, double delta, double Delta,
                  int32_t max_iter, void *d_ws, int64_t ws_bytes, int64_t *h_offsets, void *stream) {
    B3C_REQUIRE(n > 0 && 0 <= row_lo && row_lo < row_hi && row_hi <= n, "bad row block [%d,%d) of %d", row_lo, row_hi, n);
    B3C_REQUIRE(row_lo % CHUNK == 0 && (row_hi % CHUNK == 0 || row_hi == n), "row blocks must be %d-row aligned", CHUNK);
    B3C_REQUIRE(d_indptr && d_ws && h_offsets && nnz_local >= 0, "bad arguments");
    const KRLayout L = kr_layout(n, nnz_local, n);
    if (ws_bytes < L.total) {
        set_error("KR workspace too small: %lld < %lld", (long long)ws_bytes, (long long)L.total);
        return B3C_ERR_CAPACITY;
    }
    cudaStream_t s = (cudaStream_t)stream;
    KRArgs A;
    kr_bind(A, L, (char *)d_ws, n, row_lo, row_hi, nnz_local, d_indptr, d_indices, d_data);
    KRScalars S;
    kr_scalars_init(S, tol, delta, Delta, max_iter);
    S.state = KR_STATE_INNER;
    B3C_CUDA(cudaMemcpyAsync(A.ctl, &S, sizeof(S), cudaMemcpyHostToDevice, s));
    B3C_CUDA(cudaMemsetAsync(A.timers, 0, sizeof(KRTimers), s));
    B3C_CUDA(cudaMemsetAsync(A.part, 0, (size_t)L.n_chunks * 8 * P_COUNT, s));
    B3C_CUDA(cudaMemsetAsync(A.u, 0, (size_t)L.nvec * 8, s));
    int rc = kr_prepare(A, L, s);
    if (rc) return rc;
    h_offsets[0] = L.o_vec + L.nvec * 8 * 8;            // u: float64[n]
    h_offsets[1] = L.o_vec;                             // x: float64[n]
    h_offsets[2] = L.o_part;                            // partials: float64[7][n_chunks]
    h_offsets[3] = L.n_chunks;
    h_offsets[4] = L.o_ctl;
    std::lock_guard<std::mutex> g(g_krp_mu);
    g_krp[d_ws] = A;
    return B3C_OK;
}

static int krp_get(void *ws, KRArgs *A) {
    std::lock_guard<std::mutex> g(g_krp_mu);
    auto it = g_krp.find(ws);
    if (it == g_krp.end()) {
        set_error("workspace %p has no KR plan: call b3c_krp_setup first", ws);
        return B3C_ERR_ARG;
    }
    *A = it->second;
    return B3C_OK;
}

int b3c_krp_phase(void *d_ws, int32_t phase, void *stream) {
    KRArgs A;
    int rc = krp_get(d_ws, &A);
    if (rc) return rc;
    B3C_REQUIRE(phase >= KRP_INIT && phase <= KRP_UPDATE, "unknown phase %d", phase);
    if (phase == KRP_SPMV) return launch_spmv(A, (cudaStream_t)stream);
    const unsigned grid = (unsigned)(A.n_chunks < kNumSMs * 4 ? A.n_chunks : kNumSMs * 4);
    k_krp_phase<<<grid, KR_THREADS, 0, (cudaStream_t)stream>>>(A, phase);
    B3C_LAUNCH_CHECK();
    return B3C_OK;
}

int b3c_krp_scalar(void *d_ws, int32_t which, void *stream) {
    KRArgs A;
    int rc = krp_get(d_ws, &A);
    if (rc) return rc;
    B3C_REQUIRE(which >= KRS_OUTER_FIRST && which <= KRS_DECIDE, "unknown scalar step %d", which);
    k_krp_scalar<<<1, KR_THREADS, 0, (cudaStream_t)stream>>>(A, which);
    B3C_LAUNCH_CHECK();
    return B3C_OK;
}

int b3c_krp_state(void *d_ws, int64_t *h_state, void *stream) {
    KRArgs A;
    int rc = krp_get(d_ws, &A);
    if (rc) return rc;
    B3C_REQUIRE(h_state != nullptr, "null h_state");
    KRScalars S;
    B3C_CUDA(cudaMemcpyAsync(&S, A.ctl, sizeof(S), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    B3C_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    h_state[0] = S.state;
    h_state[1] = S.status;
    h_state[2] = S.n_iter;
    h_state[3] = S.k;
    h_state[4] = S.outer;
    h_state[5] = S.n_spmv;
    h_state[6] = S.zero_diag;
    return B3C_OK;
}

}  // extern "C"
