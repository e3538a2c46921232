// The cm_graph.edges text of device edge arrays (include/bin3c_b200.h: b3c_edges_text), byte for byte what the host
// writer b3c_edges_write_fmt (io_edges.cpp) prints for the same arrays.  The digits and the layout are in
// edgefmt.cuh; this file places the lines:
//   k_len        one thread per edge: its line length; one sum per block of EDGE_THREADS edges
//   scan         the exclusive scan of the block sums (scan_exclusive_i64), the total at the end: no host round trip
//   k_write      one thread per edge again: the digits and the length, a block scan for the line's offset in the
//                block, the line into shared memory at that offset; then the block's contiguous span goes to the
//                text with 16-byte stores (bytewise only at the two ends the neighbouring blocks share)
// Recomputing the digits in k_write is cheaper than storing them.  The power-of-5 tables are read from global memory
// through the read-only path (lanes with different exponents read different rows).
#include <algorithm>

#include "common.cuh"
#include "edgefmt.cuh"

namespace b3c {
namespace {

using namespace b3c_edgefmt;

constexpr int EDGE_THREADS = 256;
constexpr int SPAN_BYTES = EDGE_THREADS * MAX_LINE_BYTES;
static_assert(MAX_LINE_BYTES == B3C_EDGES_MAX_LINE_BYTES, "line bound");

struct EdgeLayout {
    int64_t n_blocks, sums_off, offs_off, tmp_off, bytes;
};

EdgeLayout edge_layout(int64_t n_edges) {
    EdgeLayout L;
    Carver c;
    L.n_blocks = ceil_div(n_edges > 0 ? n_edges : 1, EDGE_THREADS);
    L.sums_off = c.take(L.n_blocks * 8);
    L.offs_off = c.take((L.n_blocks + 1) * 8);
    L.tmp_off = c.take(scan_tmp_elems(L.n_blocks) * 8);
    L.bytes = c.cur;
    return L;
}

__device__ __forceinline__ Pow5 tables() { return Pow5{POW5_SPLIT, POW5_INV_SPLIT}; }

__device__ __forceinline__ Line measure(const int32_t *u, const int32_t *v, const double *w, int64_t i, int style) {
    return line_measure(__ldg(u + i), __ldg(v + i), __ldg(w + i), style, tables());
}

__global__ void __launch_bounds__(EDGE_THREADS) k_len(const int32_t *__restrict__ u, const int32_t *__restrict__ v,
                                                      const double *__restrict__ w, int64_t n, int style,
                                                      int64_t *__restrict__ sums) {
    __shared__ int s_w[33];
    const int64_t i = (int64_t)blockIdx.x * EDGE_THREADS + threadIdx.x;
    const int len = i < n ? measure(u, v, w, i, style).bytes() : 0;
    int tot;
    block_scan_excl<int>(len, s_w, &tot);
    if (threadIdx.x == 0) sums[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(EDGE_THREADS) k_write(const int32_t *__restrict__ u, const int32_t *__restrict__ v,
                                                        const double *__restrict__ w, int64_t n, int style, char sep,
                                                        const int64_t *__restrict__ offs, uint8_t *__restrict__ text) {
    __shared__ __align__(16) char buf[SPAN_BYTES + 16];
    __shared__ int s_w[33];
    const int64_t i = (int64_t)blockIdx.x * EDGE_THREADS + threadIdx.x;
    Line L;
    int32_t a = 0, b = 0;
    int len = 0;
    if (i < n) {
        a = __ldg(u + i);
        b = __ldg(v + i);
        L = line_measure(a, b, __ldg(w + i), style, tables());
        len = L.bytes();
    }
    int tot;
    const int at = block_scan_excl<int>(len, s_w, &tot);
    // buf[k] holds the byte at address base + k, base the 16-byte boundary at or below the block's span: the phase
    // comes from the address, so d_text may have any alignment.  Only bytes k >= shift are stored (none before d_text).
    uint8_t *const span = text + offs[blockIdx.x];
    const int shift = (int)((uintptr_t)span & 15);
    if (i < n) line_put(L, a, b, sep, style, buf + shift + at);
    __syncthreads();
    uint8_t *base = span - shift;
    const int end = shift + tot;
    for (int c = threadIdx.x; c * 16 < end; c += EDGE_THREADS) {
        const int lo = c * 16;
        if (lo >= shift && lo + 16 <= end) {
            *(uint4 *)(base + lo) = *(const uint4 *)(buf + lo);
        } else {
            for (int k = max(lo, shift); k < min(lo + 16, end); ++k) base[k] = (uint8_t)buf[k];
        }
    }
}

}  // namespace
}  // namespace b3c

using namespace b3c;

extern "C" {

int64_t b3c_edges_text_workspace_bytes(int64_t max_edges) {
    if (max_edges < 0) {
        set_error("b3c_edges_text_workspace_bytes: negative edge count");
        return B3C_ERR_ARG;
    }
    return edge_layout(max_edges).bytes;
}

int b3c_edges_text(void *d_ws, int64_t ws_bytes, const int32_t *d_u, const int32_t *d_v, const double *d_w,
                   int64_t n_edges, int32_t sep, int32_t float_style, uint8_t *d_text, int64_t text_capacity,
                   int64_t *h_bytes, void *stream) {
    B3C_REQUIRE(h_bytes != nullptr && n_edges >= 0, "b3c_edges_text: null h_bytes or negative edge count");
    B3C_REQUIRE(float_style == B3C_FLOAT_REPR || float_style == B3C_FLOAT_STR12,
                "b3c_edges_text: float_style %d is neither B3C_FLOAT_REPR nor B3C_FLOAT_STR12", float_style);
    B3C_REQUIRE(sep >= 0 && sep <= 255, "b3c_edges_text: separator %d is not a byte", sep);
    B3C_REQUIRE(n_edges <= INT64_MAX / B3C_EDGES_MAX_LINE_BYTES && text_capacity >= n_edges * B3C_EDGES_MAX_LINE_BYTES,
                "b3c_edges_text: the text buffer holds %lld bytes, %lld edges need %lld", (long long)text_capacity,
                (long long)n_edges, (long long)n_edges * B3C_EDGES_MAX_LINE_BYTES);
    *h_bytes = 0;
    if (n_edges == 0) return B3C_OK;                  // a zero-length tensor may report a null address
    B3C_REQUIRE(d_ws && d_u && d_v && d_w && d_text, "b3c_edges_text: null device pointer");
    const EdgeLayout L = edge_layout(n_edges);
    B3C_REQUIRE(ws_bytes >= L.bytes, "b3c_edges_text: workspace holds %lld bytes, needs %lld", (long long)ws_bytes,
                (long long)L.bytes);
    B3C_REQUIRE(L.n_blocks <= 0x7fffffff, "b3c_edges_text: %lld edges are too many for one call", (long long)n_edges);
    cudaStream_t s = (cudaStream_t)stream;
    uint8_t *ws = (uint8_t *)d_ws;
    int64_t *sums = (int64_t *)(ws + L.sums_off), *offs = (int64_t *)(ws + L.offs_off);
    k_len<<<(unsigned)L.n_blocks, EDGE_THREADS, 0, s>>>(d_u, d_v, d_w, n_edges, float_style, sums);
    B3C_LAUNCH_CHECK();
    const int rc = scan_exclusive_i64(sums, offs, L.n_blocks, (int64_t *)(ws + L.tmp_off), s);
    if (rc != B3C_OK) return rc;
    k_write<<<(unsigned)L.n_blocks, EDGE_THREADS, 0, s>>>(d_u, d_v, d_w, n_edges, float_style, (char)sep, offs,
                                                         d_text);
    B3C_LAUNCH_CHECK();
    B3C_CUDA(cudaMemcpyAsync(h_bytes, offs + L.n_blocks, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    B3C_CUDA(cudaStreamSynchronize(s));
    return B3C_OK;
}

}  // extern "C"
