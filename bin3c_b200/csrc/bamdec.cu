// Name-sorted BAM -> packed pair records on the device (include/bin3c_b200.h: b3c_bamdec_*).  The output is the
// output of the host reader (io_bam.cpp: next_alignment + read_pairs_impl, contact-map records only), record for
// record and in the same order, and the counters are those of b3c_bam_stats indices 0-7.
//
// The host reads the file in SLABS of whole BGZF blocks and lists the blocks (include/bin3c_io.h: b3c_bgzf_scan);
// everything else happens here, one slab at a time, in a buffer U that holds the partial record the previous slab
// ended with (the carry) followed by the inflated blocks:
//   k_inflate, k_crc   raw inflate (output size == ISIZE) and CRC-32 of every block: bgzf_inflate_blocks (bgzf.cu)
//   k_guess    one thread per block: guess where the block's first record starts (the block start when it passes the
//              field checks -- htslib flushes a block before a record that would not fit -- else the first offset
//              that does) and walk the block_size chain from there to the first record start at or after the block end
//   k_verify   one thread: walks the verified chain block to block, taking a block's exit from k_guess when its guess
//              equals the verified entry and walking the block again otherwise (a repair).  Speculation only changes
//              how much is walked, never the result.
//   k_scan     one thread per block: parses the records that start in the block (the checks and matchers of
//              next_alignment) and runs the pairing recurrence over its informative records twice, for the two ways
//              the block can be entered: its first informative record starting a pair (A) or closing one (B)
//   k_link     one thread per block: compares the block's first informative record with the previous informative
//              record (an earlier block, or the pending first mate carried from the previous slab)
//   k_chain    one thread: picks A or B per block from the incoming pending bit, sums the counters, gives every
//              block its first output index, and keeps the pending first mate for the next slab
//   k_emit     one thread per block: writes the block's records in input order
// Errors are recorded as (stream position << 8 | code) with atomicMin, so the one reported is the first in the stream.
#include "bgzf.cuh"
#include "common.cuh"

namespace b3c {
namespace {

constexpr uint32_t BAD_TID = 0x7fffffffu;
constexpr unsigned long long NO_ERR = ~0ull;

enum : int {
    E_INFLATE = 1,
    E_CRC = 2,
    E_SHORT = 3,
    E_OVERRUN = 4,
    E_UNTERM = 5,
    E_TRUNC_ARRAY = 6,
    E_MALFORMED_ARRAY = 7,
    E_UNKNOWN_TAG = 8,
    E_TRUNCATED = 9,
};

const char *err_text(int code) {
    switch (code) {
        case E_INFLATE: return "corrupt BGZF block (inflate)";
        case E_CRC: return "corrupt BGZF block (CRC mismatch)";
        case E_SHORT: return "alignment record shorter than its fixed fields";
        case E_OVERRUN: return "alignment record overruns its block size";
        case E_UNTERM: return "unterminated string tag";
        case E_TRUNC_ARRAY: return "truncated array tag";
        case E_MALFORMED_ARRAY: return "malformed array tag";
        case E_UNKNOWN_TAG: return "unknown tag type";
        case E_TRUNCATED: return "truncated alignment record";
        default: return "malformed BAM file";
    }
}

// the pending first mate, carried from one slab to the next
struct R1 {
    int32_t pending, tid, pos, flag, match, name_len;
    uint8_t name[256];
};

struct Header {
    int32_t min_mapq, strong, min_insert, n_refs;
    int64_t next_rec;                 // stream offset of the first record not yet decoded
    unsigned long long err;           // (stream offset << 8) | code of the first error, NO_ERR when none
    int64_t stats[8];                 // b3c_bam_stats indices 0-7
    int64_t result[4];                // of the last slab: records, next_rec, repaired blocks, informative records
    R1 in, out;
};

struct BlockWork {
    int64_t s, x, e;                  // guessed entry, exit from the guess, verified entry (U offsets)
    int64_t first_inf, last_inf;      // U offsets of the block's first / last informative record, -1 none
    int64_t prev_inf;                 // U offset of the informative record before first_inf, -1: the carried r1
    int64_t base;                     // first output index
    int32_t n_aln, n_inf;
    int32_t emit[2], pairs[2], shrt[2], orphan[2];
    uint8_t endp[2], same_first, short_first, variant, pad[3];
};

// the layout begin() laid out for a workspace: kept on the host so that a slab call needs no round trip
struct Layout {
    int64_t bytes;
    int32_t n_refs, max_blocks;
    int64_t tid_off, work_off;
};
std::mutex g_layout_mu;
std::unordered_map<const void *, Layout> g_layouts;

int64_t header_bytes() { return align_up(sizeof(Header), 256); }

struct Slab {
    Header *hd;
    BlockWork *work;
    const int32_t *tid2idx;
    const uint8_t *comp;
    const int64_t *blocks;            // [3 n]: c_off, bsize | isize << 32, u_off (from the first inflated byte)
    int32_t nb;
    uint8_t *u;
    int64_t carry, u_end;             // U = carry bytes, then the blocks; u_end = carry + sum ISIZE
    int64_t u0;                       // stream offset of U[0]
    int32_t last;
    uint64_t *out;
    int64_t out_cap;
};

__device__ __forceinline__ uint32_t rd32(const uint8_t *p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
__device__ __forceinline__ uint32_t rd16(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }

__device__ __forceinline__ int64_t blk_isize(const Slab &S, int b) { return (int64_t)((uint64_t)S.blocks[3 * b + 1] >> 32); }
__device__ __forceinline__ int64_t blk_bsize(const Slab &S, int b) { return S.blocks[3 * b + 1] & 0xffffffffll; }
__device__ __forceinline__ int64_t blk_lo(const Slab &S, int b) { return b == 0 ? 0 : S.carry + S.blocks[3 * b + 2]; }
__device__ __forceinline__ int64_t blk_hi(const Slab &S, int b) { return S.carry + S.blocks[3 * b + 2] + blk_isize(S, b); }

__device__ __forceinline__ void record_error(Header *hd, int64_t stream_pos, int code) {
    atomicMin(&hd->err, ((unsigned long long)stream_pos << 8) | (unsigned long long)code);
}

// the block_size chain from p until it reaches `lim`, stops at a record the buffer does not hold completely, or at a
// block_size below the fixed fields; returns where it stopped
__device__ int64_t walk(const Slab &S, int64_t p, int64_t lim) {
    while (p < lim) {
        if (p + 4 > S.u_end) break;
        const uint32_t bs = rd32(S.u + p);
        if (bs < 32 || p + 4 + (int64_t)bs > S.u_end) break;
        p += 4 + (int64_t)bs;
    }
    return p;
}

// fixed fields of a record at p that a real record has; only a guess, which the verification corrects
__device__ bool plausible_fields(const Slab &S, int64_t p) {
    if (p + 36 > S.u_end) return false;
    const uint8_t *r = S.u + p;
    const uint32_t bs = rd32(r);
    const int32_t tid = (int32_t)rd32(r + 4), pos = (int32_t)rd32(r + 8), ntid = (int32_t)rd32(r + 24);
    const uint32_t l_name = r[12], n_cig = rd16(r + 16);
    const int32_t l_seq = (int32_t)rd32(r + 20);
    if (bs < 32 || tid < -1 || pos < -1 || ntid < -1 || l_name == 0 || l_seq < 0) return false;
    if (32 + (int64_t)l_name + 4 * (int64_t)n_cig > (int64_t)bs) return false;
    if (p + 36 + (int64_t)l_name > S.u_end) return true;
    return r[36 + l_name - 1] == 0;
}

__device__ bool plausible(const Slab &S, int64_t p) {
    if (!plausible_fields(S, p)) return false;
    // the next record must pass too, so a block_size pointing past the buffer is rejected: sequence and quality bytes
    // read as a block_size are mostly huge.  (A block that starts the slab's unfinished last record is walked again.)
    const int64_t q = p + 4 + (int64_t)rd32(S.u + p);
    if (q > S.u_end) return false;
    return q + 36 > S.u_end || plausible_fields(S, q);
}

struct Rec {
    int32_t tid, pos, flag;
    bool match, inf;
    const uint8_t *name;
    int32_t name_len;
};

// next_alignment (io_bam.cpp) for the record whose block_size field is at U[p]; the caller has checked bs >= 32 and
// that the record lies inside U.  Returns 0 or an error code.
__device__ int parse_record(const Slab &S, int64_t p, uint32_t bs, Rec *a) {
    const uint8_t *b = S.u + p + 4;
    const int64_t end = bs;
    const uint32_t l_name = b[8], mapq = b[9], n_cig = rd16(b + 12);
    a->tid = (int32_t)rd32(b);
    a->pos = (int32_t)rd32(b + 4);
    a->flag = (int32_t)rd16(b + 14);
    if (32 + (int64_t)l_name + 4 * (int64_t)n_cig > end) return E_OVERRUN;
    a->name = b + 32;
    int32_t nl = 0;
    while (nl < (int32_t)l_name && b[32 + nl] != 0) ++nl;
    a->name_len = nl;
    int64_t cg = 32 + l_name;
    uint32_t n_ops = n_cig;
    const uint32_t l_seq = rd32(b + 16);
    if (n_cig == 2 && (rd32(b + cg) & 0xf) == 4 && (rd32(b + cg) >> 4) == l_seq && (rd32(b + cg + 4) & 0xf) == 3) {
        int64_t aux = cg + 8 + ((int64_t)l_seq + 1) / 2 + (int64_t)l_seq;
        while (aux + 3 <= end) {
            const uint8_t t = b[aux + 2];
            const int64_t v = aux + 3;
            int64_t len = 0;
            auto size_of = [](uint8_t c) -> int64_t {
                return (c == 'A' || c == 'c' || c == 'C') ? 1 : (c == 's' || c == 'S') ? 2 : (c == 'i' || c == 'I' || c == 'f') ? 4 : 0;
            };
            if (t == 'Z' || t == 'H') {
                int64_t z = v;
                while (z < end && b[z] != 0) ++z;
                if (z >= end) return E_UNTERM;
                len = z - v + 1;
            } else if (t == 'B') {
                if (v + 5 > end) return E_TRUNC_ARRAY;
                const int64_t es = size_of(b[v]), cnt = rd32(b + v + 1);
                if (es == 0 || v + 5 + es * cnt > end) return E_MALFORMED_ARRAY;
                if (b[aux] == 'C' && b[aux + 1] == 'G' && b[v] == 'I' && cnt > 0) {
                    cg = v + 5;
                    n_ops = (uint32_t)cnt;
                    break;
                }
                len = 5 + es * cnt;
            } else {
                len = size_of(t);
                if (len == 0) return E_UNKNOWN_TAG;
            }
            aux = v + len;
        }
    }
    bool m = (int32_t)mapq >= S.hd->min_mapq;
    if (m && S.hd->strong > 0) {
        if (n_ops == 0) {
            m = false;
        } else {
            const uint32_t op = rd32(b + cg + 4 * (int64_t)((a->flag & 0x10) ? (n_ops - 1) : 0));
            m = (op & 0xf) == 0 && (int32_t)(op >> 4) >= S.hd->strong;
        }
    }
    a->match = m;
    a->inf = (a->flag & (0x4 | 0x100 | 0x800)) == 0;
    return 0;
}

__device__ __forceinline__ bool same_name(const Rec &x, const Rec &y) {
    if (x.name_len != y.name_len) return false;
    for (int k = 0; k < x.name_len; ++k)
        if (x.name[k] != y.name[k]) return false;
    return true;
}

__device__ __forceinline__ Rec from_r1(const R1 &r) {
    Rec a;
    a.tid = r.tid;
    a.pos = r.pos;
    a.flag = r.flag;
    a.match = r.match != 0;
    a.inf = true;
    a.name = r.name;
    a.name_len = r.name_len;
    return a;
}

// the record read_pairs_impl writes for (r1, r2); *short_insert when the insert filter drops the pair instead
__device__ uint64_t pair_record(const Slab &S, const Rec &r1, const Rec &r2, bool *short_insert) {
    const int32_t n_refs = S.hd->n_refs;
    const bool in1 = r1.tid >= 0 && r1.tid < n_refs, in2 = r2.tid >= 0 && r2.tid < n_refs;
    const bool pass = r1.match && r2.match;
    *short_insert = false;
    if (S.hd->min_insert > 0 && pass && in1 && in2 && S.tid2idx[r1.tid] >= 0 && S.tid2idx[r2.tid] >= 0) {
        const bool swap = (r1.flag & 0x80) != 0;
        const int32_t f1 = swap ? r2.flag : r1.flag;
        const int32_t p1 = swap ? r2.pos : r1.pos, p2 = swap ? r1.pos : r2.pos;
        if ((f1 & 0x2) && (int64_t)p2 - (int64_t)p1 < (int64_t)S.hd->min_insert) *short_insert = true;
    }
    const uint64_t t1 = in1 ? (uint32_t)r1.tid : BAD_TID, t2 = in2 ? (uint32_t)r2.tid : BAD_TID;
    return t1 | ((uint64_t)(pass ? 1u : 0u) << 31) | (t2 << 32);
}

// parse the (complete, already checked) record at U[p]
__device__ Rec record_at(const Slab &S, int64_t p) {
    Rec a;
    parse_record(S, p, rd32(S.u + p), &a);
    return a;
}

__global__ void k_begin(Header *hd, int32_t min_mapq, int32_t strong, int32_t min_insert, int32_t n_refs, int64_t data_offset) {
    hd->min_mapq = min_mapq;
    hd->strong = strong;
    hd->min_insert = min_insert;
    hd->n_refs = n_refs;
    hd->next_rec = data_offset;
    hd->err = NO_ERR;
    for (int k = 0; k < 8; ++k) hd->stats[k] = 0;
    for (int k = 0; k < 4; ++k) hd->result[k] = 0;
    hd->in.pending = 0;
    hd->out.pending = 0;
}

__global__ void __launch_bounds__(128) k_guess(Slab S) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= S.nb) return;
    const int64_t lo = blk_lo(S, b), hi = blk_hi(S, b);
    int64_t s = -1;
    for (int64_t p = lo; p < hi; ++p)
        if (plausible(S, p)) {
            s = p;
            break;
        }
    S.work[b].s = s;
    S.work[b].x = s < 0 ? -1 : walk(S, s, hi);
}

__global__ void k_verify(Slab S) {
    int64_t e = S.hd->next_rec - S.u0, repaired = 0;
    bool stopped = false;
    for (int b = 0; b < S.nb; ++b) {
        const int64_t hi = blk_hi(S, b);
        BlockWork &w = S.work[b];
        w.e = e;
        if (stopped || e >= hi) continue;
        int64_t nx;
        if (b > 0 && e == w.s) {
            nx = w.x;
        } else {
            nx = walk(S, e, hi);
            repaired += (b > 0);
        }
        if (nx < hi) stopped = true;                   // the chain ends inside this block
        e = nx;
    }
    S.hd->next_rec = S.u0 + e;
    S.hd->result[2] = repaired;
}

// the records that start in block b, in order: calls f(p, rec) for each; records errors; false when there are none
template <typename F>
__device__ void for_each_record(const Slab &S, int b, bool report, F f) {
    const int64_t lo = blk_lo(S, b), hi = blk_hi(S, b);
    int64_t p = S.work[b].e;
    if (p < lo || p >= hi) return;
    while (p < hi) {
        if (p + 4 > S.u_end) {
            if (report && S.last) record_error(S.hd, S.u0 + p, E_TRUNCATED);
            return;
        }
        const uint32_t bs = rd32(S.u + p);
        if (bs < 32) {
            if (report) record_error(S.hd, S.u0 + p, E_SHORT);
            return;
        }
        if (p + 4 + (int64_t)bs > S.u_end) {
            if (report && S.last) record_error(S.hd, S.u0 + p, E_TRUNCATED);
            return;
        }
        Rec a;
        const int rc = parse_record(S, p, bs, &a);
        if (rc) {
            if (report) record_error(S.hd, S.u0 + p, rc);
            return;
        }
        f(p, a);
        p += 4 + (int64_t)bs;
    }
}

__global__ void __launch_bounds__(128) k_scan(Slab S) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= S.nb) return;
    int32_t n_aln = 0, n_inf = 0;
    int64_t first = -1, last = -1;
    int pend[2] = {1, 0};                              // A: the first informative record is pending; B: it closed a pair
    int32_t emit[2] = {0, 0}, pairs[2] = {0, 0}, shrt[2] = {0, 0}, orphan[2] = {0, 0};
    Rec prev;
    prev.name_len = 0;
    prev.name = nullptr;
    for_each_record(S, b, true, [&](int64_t p, const Rec &a) {
        ++n_aln;
        if (!a.inf) return;
        ++n_inf;
        if (first < 0) {
            first = p;
        } else {
            const bool same = same_name(prev, a);
            for (int v = 0; v < 2; ++v) {
                if (pend[v] && same) {
                    bool sh;
                    pair_record(S, prev, a, &sh);
                    pairs[v] += 1;
                    if (sh) shrt[v] += 1;
                    else emit[v] += 1;
                    pend[v] = 0;
                } else {
                    if (pend[v]) orphan[v] += 1;
                    pend[v] = 1;
                }
            }
        }
        last = p;
        prev = a;
    });
    BlockWork &w = S.work[b];
    w.n_aln = n_aln;
    w.n_inf = n_inf;
    w.first_inf = first;
    w.last_inf = last;
    for (int v = 0; v < 2; ++v) {
        w.emit[v] = emit[v];
        w.pairs[v] = pairs[v];
        w.shrt[v] = shrt[v];
        w.orphan[v] = orphan[v];
        w.endp[v] = (uint8_t)pend[v];
    }
}

__global__ void __launch_bounds__(128) k_link(Slab S) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= S.nb) return;
    BlockWork &w = S.work[b];
    w.same_first = 0;
    w.short_first = 0;
    w.prev_inf = -1;
    if (w.n_inf == 0) return;
    int64_t prev = -1;
    for (int k = b - 1; k >= 0; --k)
        if (S.work[k].n_inf > 0) {
            prev = S.work[k].last_inf;
            break;
        }
    w.prev_inf = prev;
    Rec r1;
    if (prev >= 0) r1 = record_at(S, prev);
    else if (S.hd->in.pending) r1 = from_r1(S.hd->in);
    else return;                                       // nothing pending: the first record starts a pair whatever its name
    const Rec r2 = record_at(S, w.first_inf);
    if (!same_name(r1, r2)) return;
    w.same_first = 1;
    bool sh;
    pair_record(S, r1, r2, &sh);
    w.short_first = sh ? 1 : 0;
}

__global__ void k_chain(Slab S) {
    Header *hd = S.hd;
    int64_t *st = hd->stats;
    int s = hd->in.pending;
    int64_t base = 0, inf = 0;
    int last_blk = -1;
    for (int b = 0; b < S.nb; ++b) {
        BlockWork &w = S.work[b];
        st[5] += 1;
        st[6] += blk_bsize(S, b) + 1;
        st[7] += blk_isize(S, b);
        st[0] += w.n_aln;
        st[1] += w.n_inf;
        inf += w.n_inf;
        w.base = base;
        if (w.n_inf == 0) {
            w.variant = 0xff;
            continue;
        }
        int v;
        if (s && w.same_first) {
            v = 1;
            st[2] += 1;
            if (w.short_first) st[3] += 1;
            else base += 1;
        } else {
            v = 0;
            if (s) st[4] += 1;                         // the pending record never found its mate
        }
        w.variant = (uint8_t)v;
        st[2] += w.pairs[v];
        st[3] += w.shrt[v];
        st[4] += w.orphan[v];
        base += w.emit[v];
        s = w.endp[v];
        last_blk = b;
    }
    // the pending first mate for the next slab
    if (last_blk < 0) {
        hd->out = hd->in;
    } else if (s) {
        const Rec a = record_at(S, S.work[last_blk].last_inf);
        R1 &o = hd->out;
        o.pending = 1;
        o.tid = a.tid;
        o.pos = a.pos;
        o.flag = a.flag;
        o.match = a.match ? 1 : 0;
        o.name_len = a.name_len;
        for (int k = 0; k < a.name_len; ++k) o.name[k] = a.name[k];
    } else {
        hd->out.pending = 0;
    }
    if (S.last && hd->next_rec < S.u0 + S.u_end)
        record_error(hd, hd->next_rec, E_TRUNCATED);   // the file ends inside a record
    if (S.last && hd->out.pending) {
        st[4] += 1;                                    // StopIteration with a mate pending
        hd->out.pending = 0;
    }
    hd->result[0] = base;
    hd->result[1] = hd->next_rec;
    if (S.nb == 0) hd->result[2] = 0;
    hd->result[3] = inf;
}

__global__ void __launch_bounds__(128) k_emit(Slab S) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= S.nb) return;
    const BlockWork &w = S.work[b];
    if (w.variant > 1) return;
    int64_t idx = w.base;
    bool first = true;
    int pend = 0;
    Rec prev;
    prev.name_len = 0;
    prev.name = nullptr;
    for_each_record(S, b, false, [&](int64_t p, const Rec &a) {
        if (!a.inf) return;
        bool same = false, sh = false;
        if (first) {
            first = false;
            if (w.variant == 1) {
                const Rec r1 = w.prev_inf >= 0 ? record_at(S, w.prev_inf) : from_r1(S.hd->in);
                const uint64_t r = pair_record(S, r1, a, &sh);
                if (!sh && idx < S.out_cap) S.out[idx] = r;
                idx += sh ? 0 : 1;
                pend = 0;
            } else {
                pend = 1;
            }
        } else {
            same = same_name(prev, a);
            if (pend && same) {
                const uint64_t r = pair_record(S, prev, a, &sh);
                if (!sh && idx < S.out_cap) S.out[idx] = r;
                idx += sh ? 0 : 1;
                pend = 0;
            } else {
                pend = 1;
            }
        }
        prev = a;
    });
}

__global__ void k_finish(Header *hd) { hd->in = hd->out; }

}  // namespace
}  // namespace b3c

using namespace b3c;

extern "C" {

int64_t b3c_bamdec_workspace_bytes(int32_t max_blocks, int32_t n_refs) {
    if (max_blocks < 1 || n_refs < 0) {
        set_error("b3c_bamdec_workspace_bytes: max_blocks must be positive and n_refs non-negative");
        return B3C_ERR_ARG;
    }
    return header_bytes() + align_up(4 * (int64_t)n_refs, 256) + (int64_t)max_blocks * (int64_t)sizeof(BlockWork);
}

int b3c_bamdec_begin(void *d_ws, int64_t ws_bytes, int32_t min_mapq, int32_t strong, int32_t min_insert,
                     const int32_t *d_tid2idx, int32_t n_refs, int64_t data_offset, void *stream) {
    B3C_REQUIRE(d_ws != nullptr, "b3c_bamdec_begin: null workspace");
    B3C_REQUIRE(n_refs >= 0 && data_offset >= 0, "b3c_bamdec_begin: negative n_refs or data offset");
    B3C_REQUIRE(min_insert <= 0 || d_tid2idx != nullptr, "b3c_bamdec_begin: min_insert needs the tid -> index table");
    const int64_t fixed = header_bytes() + align_up(4 * (int64_t)n_refs, 256);
    B3C_REQUIRE(ws_bytes >= fixed + (int64_t)sizeof(BlockWork), "b3c_bamdec_begin: workspace too small");
    cudaStream_t s = (cudaStream_t)stream;
    Layout L;
    L.bytes = ws_bytes;
    L.n_refs = n_refs;
    L.tid_off = header_bytes();
    L.work_off = fixed;
    const int64_t mb = (ws_bytes - fixed) / (int64_t)sizeof(BlockWork);
    L.max_blocks = (int32_t)(mb > 0x7fffffff ? 0x7fffffff : mb);
    if (d_tid2idx && n_refs > 0)
        B3C_CUDA(cudaMemcpyAsync((uint8_t *)d_ws + L.tid_off, d_tid2idx, 4 * (size_t)n_refs, cudaMemcpyDeviceToDevice, s));
    k_begin<<<1, 1, 0, s>>>((Header *)d_ws, min_mapq, strong < 0 ? 0 : strong, min_insert < 0 ? 0 : min_insert, n_refs,
                            data_offset);
    B3C_LAUNCH_CHECK();
    std::lock_guard<std::mutex> g(g_layout_mu);
    g_layouts[d_ws] = L;
    return B3C_OK;
}

int b3c_bamdec_slab(void *d_ws, const uint8_t *d_comp, const int64_t *d_blocks, int32_t n_blocks, int64_t stream_offset,
                    int64_t u_bytes, const uint8_t *d_carry, int64_t carry_bytes, uint8_t *d_u, int64_t u_capacity,
                    int32_t last, uint64_t *d_out, int64_t out_capacity, int64_t *h_result, void *stream) {
    Layout L;
    {
        std::lock_guard<std::mutex> g(g_layout_mu);
        auto it = g_layouts.find(d_ws);
        B3C_REQUIRE(it != g_layouts.end(), "b3c_bamdec_slab: call b3c_bamdec_begin on this workspace first");
        L = it->second;
    }
    B3C_REQUIRE(n_blocks >= 0 && n_blocks <= L.max_blocks, "b3c_bamdec_slab: %d blocks, the workspace holds %d", n_blocks,
                L.max_blocks);
    B3C_REQUIRE(h_result != nullptr && (n_blocks == 0 || (d_comp && d_blocks)), "b3c_bamdec_slab: null argument");
    B3C_REQUIRE(carry_bytes >= 0 && u_bytes >= 0 && stream_offset >= carry_bytes && (carry_bytes == 0 || d_carry),
                "b3c_bamdec_slab: bad carry");
    B3C_REQUIRE(d_u != nullptr && u_capacity >= carry_bytes + u_bytes, "b3c_bamdec_slab: U holds %lld bytes, needs %lld",
                (long long)u_capacity, (long long)(carry_bytes + u_bytes));
    B3C_REQUIRE(out_capacity >= 0 && (out_capacity == 0 || d_out), "b3c_bamdec_slab: null output");
    cudaStream_t s = (cudaStream_t)stream;
    if (carry_bytes > 0) B3C_CUDA(cudaMemcpyAsync(d_u, d_carry, (size_t)carry_bytes, cudaMemcpyDeviceToDevice, s));
    Slab S;
    S.hd = (Header *)d_ws;
    S.work = (BlockWork *)((uint8_t *)d_ws + L.work_off);
    S.tid2idx = (const int32_t *)((uint8_t *)d_ws + L.tid_off);
    S.comp = d_comp;
    S.blocks = d_blocks;
    S.nb = n_blocks;
    S.u = d_u;
    S.carry = carry_bytes;
    S.u_end = carry_bytes + u_bytes;
    S.u0 = stream_offset - carry_bytes;
    S.last = last ? 1 : 0;
    S.out = d_out;
    S.out_cap = out_capacity;
    if (n_blocks > 0) {
        const int g128 = (int)ceil_div(n_blocks, 128);
        BgzfBlocks B;
        B.comp = d_comp;
        B.blocks = d_blocks;
        B.nb = n_blocks;
        B.u = d_u + carry_bytes;
        B.u_cap = u_bytes;
        B.err = &S.hd->err;
        B.err_base = S.u0 + carry_bytes;
        B.e_inflate = E_INFLATE;
        B.e_crc = E_CRC;
        const int rc = bgzf_inflate_blocks(B, s);
        if (rc != B3C_OK) return rc;
        k_guess<<<g128, 128, 0, s>>>(S);
        B3C_LAUNCH_CHECK();
        k_verify<<<1, 1, 0, s>>>(S);
        B3C_LAUNCH_CHECK();
        k_scan<<<g128, 128, 0, s>>>(S);
        B3C_LAUNCH_CHECK();
        k_link<<<g128, 128, 0, s>>>(S);
        B3C_LAUNCH_CHECK();
    }
    // with no blocks, the chain still closes the file (a pending first mate at the end is unpaired)
    k_chain<<<1, 1, 0, s>>>(S);
    B3C_LAUNCH_CHECK();
    if (n_blocks > 0) {
        k_emit<<<(int)ceil_div(n_blocks, 128), 128, 0, s>>>(S);
        B3C_LAUNCH_CHECK();
    }
    k_finish<<<1, 1, 0, s>>>(S.hd);
    B3C_LAUNCH_CHECK();
    struct {
        int64_t result[4];
        unsigned long long err;
    } r;
    B3C_CUDA(cudaMemcpyAsync(r.result, S.hd->result, sizeof(r.result), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaMemcpyAsync(&r.err, &S.hd->err, sizeof(r.err), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaStreamSynchronize(s));
    for (int k = 0; k < 4; ++k) h_result[k] = r.result[k];
    if (r.err != NO_ERR) {
        set_error("%s at uncompressed stream offset %llu", err_text((int)(r.err & 0xff)), r.err >> 8);
        return B3C_ERR_FORMAT;
    }
    if (r.result[0] > out_capacity) {
        set_error("b3c_bamdec_slab: %lld records, the output holds %lld", (long long)r.result[0], (long long)out_capacity);
        return B3C_ERR_CAPACITY;
    }
    return B3C_OK;
}

int b3c_bamdec_stats(const void *d_ws, int64_t *h_stats, int32_t n_stats, void *stream) {
    B3C_REQUIRE(d_ws != nullptr && h_stats != nullptr && n_stats >= 0, "b3c_bamdec_stats: null argument");
    int64_t v[8];
    cudaStream_t s = (cudaStream_t)stream;
    B3C_CUDA(cudaMemcpyAsync(v, ((const Header *)d_ws)->stats, sizeof(v), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaStreamSynchronize(s));
    for (int k = 0; k < n_stats && k < 8; ++k) h_stats[k] = v[k];
    return B3C_OK;
}

}  // extern "C"
