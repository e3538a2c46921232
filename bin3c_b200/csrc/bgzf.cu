// BGZF-framed gzip on the device (include/bin3c_b200.h: b3c_bgzf_*), and the block inflate the BAM decoder shares.
//
// Deflate, one CTA of DEFLATE_THREADS threads per member, the member's input in shared memory:
//   k_deflate  load the input; warp 0 builds the hash chains 32 positions a step (__match_any_sync finds the lanes of a
//              step with the same hash: a lane's chain link is the nearest lower such lane, else the bucket head) while
//              warp 1 takes the CRC-32; every thread finds the matches of one position per tile (tiles from the end of
//              the member down, so that a tile overwrites chain links no later tile reads with the match lengths);
//              one thread parses (deflate.cuh: parse); histograms by shared-memory atomics over per-thread segments;
//              one thread plans the codes; a block scan of the segments' bit counts places each segment, and every
//              thread writes its tokens into the member's payload slot (32-bit words, OR-ed: neighbours share words)
//   scan       the exclusive scan of the member sizes (scan_exclusive_i64): where each member goes
//   k_pack     one CTA per member: BGZF header, payload and trailer at the member's offset
// The output is byte for byte what deflate_member() of deflate.cuh writes on the host.
#include "bgzf.cuh"
#include "deflate.cuh"
#include "inflate.cuh"

namespace b3c {
namespace {

using namespace b3c_deflate;

constexpr int DEFLATE_THREADS = 512;
constexpr unsigned long long NO_ERR = ~0ull;

__device__ __forceinline__ uint32_t rd32(const uint8_t *p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

__device__ __forceinline__ void crc_table(uint32_t *table) {
    for (int k = threadIdx.x; k < 256; k += blockDim.x) {
        uint32_t c = (uint32_t)k;
        for (int j = 0; j < 8; ++j) c = (c & 1) ? (c >> 1) ^ b3c_inflate::CRC_POLY : c >> 1;
        table[k] = c;
    }
}

// CRC-32 of data[0, n) by one warp: 32 lane pieces joined in order, crc(A || B) = crc(A) * x^(8 len B) + crc(B);
// the result is valid in lane 0
__device__ uint32_t warp_crc32(const uint32_t *table, const uint8_t *data, int64_t n) {
    const unsigned lane = lane_id();
    const int64_t piece = (n + 31) / 32;
    const int64_t lo = min((int64_t)lane * piece, n), hi = min(lo + piece, n);
    uint32_t c = ~0u;
    for (int64_t k = lo; k < hi; ++k) c = table[(c ^ data[k]) & 0xff] ^ (c >> 8);
    c = ~c;
    const uint32_t step = b3c_inflate::x8nmodp(piece);
    uint32_t joined = 0;
    for (int l = 0; l < 32; ++l) {
        const uint32_t cl = __shfl_sync(kFullMask, c, l);
        const int64_t llo = min((int64_t)l * piece, n), lhi = min(llo + piece, n);
        if (lane == 0) {
            if (l == 0) joined = cl;
            else if (lhi - llo == piece) joined = b3c_inflate::multmodp(step, joined) ^ cl;
            else joined = b3c_inflate::crc32_combine(joined, cl, lhi - llo);
        }
    }
    return joined;
}

// ---- inflate (bamdec.cu and b3c_bgzf_inflate) ----------------------------------------------------------------------

__device__ __forceinline__ int64_t blk_isize(const BgzfBlocks &B, int b) { return (int64_t)((uint64_t)B.blocks[3 * b + 1] >> 32); }
__device__ __forceinline__ int64_t blk_bsize(const BgzfBlocks &B, int b) { return B.blocks[3 * b + 1] & 0xffffffffll; }

__device__ __forceinline__ void record_error(const BgzfBlocks &B, int b, int code) {
    atomicMin(B.err, ((unsigned long long)(B.err_base + B.blocks[3 * b + 2]) << 8) | (unsigned long long)code);
}

__global__ void __launch_bounds__(64) k_inflate(BgzfBlocks B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B.nb) return;
    const int64_t isize = blk_isize(B, b);
    if (isize == 0) return;                            // the host reader does not inflate an empty block either
    const int64_t bsize = blk_bsize(B, b), u_off = B.blocks[3 * b + 2];
    if (u_off < 0 || u_off + isize > B.u_cap) {
        record_error(B, b, B.e_inflate);
        return;
    }
    const uint8_t *blk = B.comp + B.blocks[3 * b];
    const int64_t xlen = blk[10] | (blk[11] << 8);
    const int64_t plen = bsize + 1 - 12 - xlen - 8;
    int64_t n = 0;
    const int rc = b3c_inflate::inflate_raw(blk + 12 + xlen, plen, B.u + u_off, isize, &n);
    if (rc != b3c_inflate::OK || n != isize) record_error(B, b, B.e_inflate);
}

__global__ void __launch_bounds__(256) k_crc(BgzfBlocks B) {
    __shared__ uint32_t table[256];
    crc_table(table);
    __syncthreads();
    const int b = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (b >= B.nb) return;
    const int64_t isize = blk_isize(B, b), u_off = B.blocks[3 * b + 2];
    if (isize == 0 || u_off < 0 || u_off + isize > B.u_cap) return;
    const uint32_t joined = warp_crc32(table, B.u + u_off, isize);
    if (lane_id() == 0) {
        const uint8_t *blk = B.comp + B.blocks[3 * b];
        if (joined != rd32(blk + blk_bsize(B, b) + 1 - 8)) record_error(B, b, B.e_crc);
    }
}

// ---- deflate -------------------------------------------------------------------------------------------------------

struct __align__(16) DeflateShared {
    uint8_t in[MEMBER_INPUT + 16];
    uint16_t prev[MEMBER_INPUT];      // hash chains, then match lengths, then tokens
    union {
        uint16_t head[HASH_SIZE];     // the chain phase
        struct {
            uint32_t lfreq[LCODES], dfreq[DCODES];
            Dyn D;
        } t;                          // after it
    } u;
    uint32_t crc[256];
    int scan[33];
    long long bits;
    int stored;
};

__global__ void __launch_bounds__(DEFLATE_THREADS, 1)
    k_deflate(const uint8_t *__restrict__ in_all, int64_t n_all, uint16_t *__restrict__ dist_all,
              uint32_t *__restrict__ payload_all, int64_t *__restrict__ sizes, uint32_t *__restrict__ crcs) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    DeflateShared &S = *reinterpret_cast<DeflateShared *>(smem_raw);
    const int m = blockIdx.x, t = threadIdx.x;
    const int64_t lo = (int64_t)m * MEMBER_INPUT;
    const int n = (int)min((int64_t)MEMBER_INPUT, n_all - lo);
    uint16_t *dist = dist_all + lo;
    uint32_t *words = payload_all + (int64_t)m * (MEMBER_MAX / 4);
    for (int k = t; k < n; k += DEFLATE_THREADS) S.in[k] = in_all[lo + k];
    for (int k = t; k < HASH_SIZE; k += DEFLATE_THREADS) S.u.head[k] = NONE;
    crc_table(S.crc);
    __syncthreads();

    const int warp = t >> 5, lane = t & 31;
    if (warp == 0) {
        for (int base = 0; base < n; base += 32) {
            const int i = base + lane;
            const bool has = i + MIN_MATCH <= n;
            const uint32_t h = has ? hash3(S.in + i) : (uint32_t)(HASH_SIZE + lane);
            const unsigned peers = __match_any_sync(kFullMask, h);
            const unsigned lower = peers & lanemask_lt();
            uint16_t p = NONE;
            if (has) p = lower ? (uint16_t)(base + 31 - __clz(lower)) : S.u.head[h];
            if (i < n) S.prev[i] = p;
            __syncwarp();
            if (has && lane == 31 - __clz(peers)) S.u.head[h] = (uint16_t)i;
            __syncwarp();
        }
    } else if (warp == 1) {
        const uint32_t c = warp_crc32(S.crc, S.in, n);
        if (lane == 0) crcs[m] = c;
    }
    __syncthreads();

    for (int base = n > 0 ? (n - 1) / DEFLATE_THREADS * DEFLATE_THREADS : -1; base >= 0; base -= DEFLATE_THREADS) {
        const int i = base + t;
        int l = 0, d = 0;
        if (i < n) {
            l = find_match(S.in, n, S.prev, i, &d);
            dist[i] = (uint16_t)d;
        }
        __syncthreads();                               // every read of this tile's chain links is done
        if (i < n) S.prev[i] = (uint16_t)l;
        __syncthreads();
    }

    for (int k = t; k < LCODES; k += DEFLATE_THREADS) S.u.t.lfreq[k] = 0;
    for (int k = t; k < DCODES; k += DEFLATE_THREADS) S.u.t.dfreq[k] = 0;
    if (t == 0) parse(S.prev, n);
    __syncthreads();
    const int seg = (n + DEFLATE_THREADS - 1) / DEFLATE_THREADS;
    const int s_lo = min(n, t * seg), s_hi = min(n, s_lo + seg);
    for (int i = s_lo; i < s_hi; ++i)
        if (S.prev[i] & TOKEN) {
            atomicAdd(&S.u.t.lfreq[token_lsym(S.in, S.prev, i)], 1u);
            if (S.prev[i] & 0x7fff) atomicAdd(&S.u.t.dfreq[dist_code(dist[i])], 1u);
        }
    __syncthreads();
    if (t == 0) {
        S.u.t.lfreq[256] = 1;
        S.bits = plan_dynamic(S.u.t.lfreq, S.u.t.dfreq, S.u.t.D);
        S.stored = use_stored(S.bits, n) ? 1 : 0;
    }
    __syncthreads();

    const Dyn &D = S.u.t.D;
    if (S.stored) {
        uint8_t *payload = reinterpret_cast<uint8_t *>(words);
        if (t == 0) {
            put_stored_head(payload, n);
            sizes[m] = HEADER_BYTES + STORED_OVERHEAD + n + TRAILER_BYTES;
        }
        for (int k = t; k < n; k += DEFLATE_THREADS) payload[STORED_OVERHEAD + k] = S.in[k];
        return;
    }
    int mine = 0;
    for (int i = s_lo; i < s_hi; ++i)
        if (S.prev[i] & TOKEN) mine += token_bits(D, S.in, S.prev, dist, i);
    int tot;
    const int off = block_scan_excl<int>(mine, S.scan, &tot);
    const int64_t nwords = (S.bits + 31) / 32;
    for (int64_t k = t; k < nwords; k += DEFLATE_THREADS) words[k] = 0;
    __syncthreads();
    BitWriter bw;
    if (t == 0) {
        bw.begin(words, 0);
        put_header(bw, D);
        bw.end();
        sizes[m] = HEADER_BYTES + (S.bits + 7) / 8 + TRAILER_BYTES;
    }
    bw.begin(words, D.header_bits + off);
    for (int i = s_lo; i < s_hi; ++i)
        if (S.prev[i] & TOKEN) put_token(bw, D, S.in, S.prev, dist, i);
    if (t == DEFLATE_THREADS - 1) bw.put(D.lcode[256], D.llen[256]);
    bw.end();
}

__global__ void __launch_bounds__(256) k_pack(const uint32_t *__restrict__ payload_all, const int64_t *__restrict__ sizes,
                                              const int64_t *__restrict__ offs, const uint32_t *__restrict__ crcs,
                                              int64_t n_all, uint8_t *__restrict__ out) {
    const int m = blockIdx.x;
    const int size = (int)sizes[m], plen = size - HEADER_BYTES - TRAILER_BYTES;
    const uint8_t *src = reinterpret_cast<const uint8_t *>(payload_all + (int64_t)m * (MEMBER_MAX / 4));
    uint8_t *dst = out + offs[m];
    for (int k = threadIdx.x; k < plen; k += blockDim.x) dst[HEADER_BYTES + k] = src[k];
    if (threadIdx.x == 0) {
        put_member_header(dst, size);
        put_u32(dst + HEADER_BYTES + plen, crcs[m]);
        put_u32(dst + HEADER_BYTES + plen + 4, (uint32_t)min((int64_t)MEMBER_INPUT, n_all - (int64_t)m * MEMBER_INPUT));
    }
}

struct DeflateLayout {
    int64_t dist_off, payload_off, sizes_off, offs_off, crc_off, tmp_off, bytes;
};

DeflateLayout deflate_layout(int64_t members) {
    DeflateLayout L;
    Carver c;
    L.dist_off = c.take(members * MEMBER_INPUT * 2);
    L.payload_off = c.take(members * MEMBER_MAX);
    L.sizes_off = c.take(members * 8);
    L.offs_off = c.take((members + 1) * 8);
    L.crc_off = c.take(members * 4);
    L.tmp_off = c.take(scan_tmp_elems(members) * 8);
    L.bytes = c.cur;
    return L;
}

}  // namespace

int bgzf_inflate_blocks(const BgzfBlocks &B, cudaStream_t s) {
    if (B.nb <= 0) return B3C_OK;
    k_inflate<<<(unsigned)ceil_div(B.nb, 64), 64, 0, s>>>(B);
    B3C_LAUNCH_CHECK();
    k_crc<<<(unsigned)ceil_div(B.nb, 8), 256, 0, s>>>(B);
    B3C_LAUNCH_CHECK();
    return B3C_OK;
}

}  // namespace b3c

using namespace b3c;

extern "C" {

int64_t b3c_bgzf_deflate_workspace_bytes(int64_t max_members) {
    if (max_members < 1 || max_members > 0x7fffffff) {
        set_error("b3c_bgzf_deflate_workspace_bytes: max_members must be in [1, 2^31)");
        return B3C_ERR_ARG;
    }
    return deflate_layout(max_members).bytes;
}

int b3c_bgzf_deflate(void *d_ws, int64_t ws_bytes, const uint8_t *d_in, int64_t n_bytes, uint8_t *d_out,
                     int64_t out_capacity, int64_t *h_out_bytes, void *stream) {
    static_assert(MEMBER_INPUT == B3C_BGZF_MEMBER_INPUT && MEMBER_MAX == B3C_BGZF_MEMBER_MAX, "member sizes");
    B3C_REQUIRE(h_out_bytes != nullptr && n_bytes >= 0, "b3c_bgzf_deflate: null h_out_bytes or negative length");
    *h_out_bytes = 0;
    if (n_bytes == 0) return B3C_OK;
    const int64_t members = ceil_div(n_bytes, MEMBER_INPUT);
    B3C_REQUIRE(members <= 0x7fffffff, "b3c_bgzf_deflate: %lld bytes are too many for one call", (long long)n_bytes);
    B3C_REQUIRE(d_ws && d_in && d_out, "b3c_bgzf_deflate: null device pointer");
    const DeflateLayout L = deflate_layout(members);
    B3C_REQUIRE(ws_bytes >= L.bytes, "b3c_bgzf_deflate: workspace holds %lld bytes, needs %lld", (long long)ws_bytes,
                (long long)L.bytes);
    B3C_REQUIRE(out_capacity >= members * MEMBER_MAX, "b3c_bgzf_deflate: the output holds %lld bytes, %lld members "
                "need %lld", (long long)out_capacity, (long long)members, (long long)(members * MEMBER_MAX));
    cudaStream_t s = (cudaStream_t)stream;
    uint8_t *ws = (uint8_t *)d_ws;
    uint16_t *dist = (uint16_t *)(ws + L.dist_off);
    uint32_t *payload = (uint32_t *)(ws + L.payload_off), *crcs = (uint32_t *)(ws + L.crc_off);
    int64_t *sizes = (int64_t *)(ws + L.sizes_off), *offs = (int64_t *)(ws + L.offs_off);
    const int smem = (int)sizeof(DeflateShared);
    B3C_CUDA(cudaFuncSetAttribute(k_deflate, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    k_deflate<<<(unsigned)members, DEFLATE_THREADS, smem, s>>>(d_in, n_bytes, dist, payload, sizes, crcs);
    B3C_LAUNCH_CHECK();
    const int rc = scan_exclusive_i64(sizes, offs, members, (int64_t *)(ws + L.tmp_off), s);
    if (rc != B3C_OK) return rc;
    k_pack<<<(unsigned)members, 256, 0, s>>>(payload, sizes, offs, crcs, n_bytes, d_out);
    B3C_LAUNCH_CHECK();
    B3C_CUDA(cudaMemcpyAsync(h_out_bytes, offs + members, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaStreamSynchronize(s));
    return B3C_OK;
}

int b3c_bgzf_inflate(void *d_ws, int64_t ws_bytes, const uint8_t *d_comp, const int64_t *d_blocks, int32_t n_blocks,
                     uint8_t *d_out, int64_t out_capacity, void *stream) {
    B3C_REQUIRE(d_ws != nullptr && ws_bytes >= 8, "b3c_bgzf_inflate: the workspace needs 8 bytes");
    B3C_REQUIRE(n_blocks >= 0 && (n_blocks == 0 || (d_comp && d_blocks)), "b3c_bgzf_inflate: null argument");
    B3C_REQUIRE(out_capacity >= 0 && (out_capacity == 0 || d_out), "b3c_bgzf_inflate: null output");
    if (n_blocks == 0) return B3C_OK;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long *err = (unsigned long long *)d_ws;
    B3C_CUDA(cudaMemsetAsync(err, 0xff, sizeof(*err), s));
    BgzfBlocks B;
    B.comp = d_comp;
    B.blocks = d_blocks;
    B.nb = n_blocks;
    B.u = d_out;
    B.u_cap = out_capacity;
    B.err = err;
    B.err_base = 0;
    B.e_inflate = 1;
    B.e_crc = 2;
    const int rc = bgzf_inflate_blocks(B, s);
    if (rc != B3C_OK) return rc;
    unsigned long long h_err = NO_ERR;
    B3C_CUDA(cudaMemcpyAsync(&h_err, err, sizeof(h_err), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaStreamSynchronize(s));
    if (h_err != NO_ERR) {
        set_error("corrupt BGZF member (%s) at uncompressed offset %llu",
                  (h_err & 0xff) == 2 ? "CRC-32 mismatch" : "does not inflate to its ISIZE", h_err >> 8);
        return B3C_ERR_FORMAT;
    }
    return B3C_OK;
}

}  // extern "C"
