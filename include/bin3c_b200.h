/*
 * bin3c_b200 -- C ABI of the B200-native bin3C contact-map hot path.
 *
 * The reference (cerebis/bin3C @ 76ad2a9) is pure Python and has no FFI layer; the
 * functions below are what a ctypes binding inside mzd/sparse_utils.py and
 * mzd/contact_map.py would call in place of the cited Python code (see INTEGRATION.md
 * for that binding).  Every entry point takes plain pointers and sizes.
 *
 * Conventions
 *   - Pointers named d_* are DEVICE pointers (e.g. torch.Tensor.data_ptr()); h_* are host
 *     pointers.  `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *   - All functions return 0 on success or a negative b3c_status; b3c_last_error()
 *     returns a thread-local message for the last failure.
 *   - No function allocates device memory: callers supply outputs and a workspace whose
 *     size comes from the matching *_workspace_bytes() query.  Entry points that hand a
 *     size back to the host (b3c_accum_reduce, b3c_kr_run, b3c_compress_count)
 *     synchronise the stream; the rest only enqueue work.
 *   - Sparse matrices are CSR: int64 indptr[n+1], int32 indices[nnz], values.
 *
 * Packed pair record (uint64, little endian) -- the input of the path, one per usable
 * read pair of the name-sorted BAM (contact_map.py:720-731):
 *     bits  0..30  BAM reference id of mate 1      (r1.reference_id)
 *     bit   31     pass flag: both mates satisfy the matcher (contact_map.py:612-622,737)
 *     bits 32..62  BAM reference id of mate 2      (r2.reference_id)
 *     bit   63     reserved, must be 0
 */
#ifndef BIN3C_B200_H
#define BIN3C_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    B3C_OK = 0,
    B3C_ERR_ARG = -1,        /* bad argument (AssertionError in the reference)          */
    B3C_ERR_CUDA = -2,       /* CUDA runtime failure                                    */
    B3C_ERR_CAPACITY = -3,   /* caller-supplied buffer or workspace too small           */
    B3C_ERR_NOCONV = -4,     /* KR: n_iter > max_iter (RuntimeError, sparse_utils.py:213) */
    B3C_ERR_NAN = -5,        /* KR: scale vector developed NaNs (sparse_utils.py:192)   */
    B3C_ERR_TIE = -6,        /* KR: max(ynew) == Delta exactly (ValueError, Q13, sparse_utils.py:179-181) */
    B3C_ERR_FORMAT = -7      /* BAM decoder: malformed file (ValueError, as the host reader raises)  */
} b3c_status;

int b3c_version(void);
const char *b3c_last_error(void);
/* number of kernels this library has launched in the calling process (bench "gpu_launches") */
int64_t b3c_launch_count(void);

/* ------------------------------------------------------------------------------------
 * Pair accumulation.  Replaces the per-pair loop of ContactMap._bin_map
 * (contact_map.py:720-798), ContactMap.make_reverse_index (contact_map.py:818-832, as the
 * dense table d_tid2idx) and Sparse2DAccumulator + get_coo (sparse_utils.py:227-266).
 *
 *   begin      once per reference table: lay out the workspace, build the tid->index rank table
 *              and zero the accumulator
 *   reset      zero the accumulator for another map over the same reference table
 *   add_pairs  classify a chunk of packed records: reference-exclusion test, then the
 *              matcher bit (filter order Q12), canonicalise i<=j, count diagonal pairs
 *              directly and append off-diagonal keys (i<<32|j).  May be called many
 *              times (streaming chunks, overlapping H2D copies).
 *   add_pairs_packed  the same for NARROW records, which make the host->device copy (what bounds the
 *              end-to-end rate) 5/8 or 6/8 of the size: bytes_per_record B = 5, 6 or 8, record =
 *              B little-endian bytes holding tid1 in bits [0, tb), the pass flag in bit tb and tid2 in
 *              bits [tb+1, 2tb+1), tb = (8B-1)/2 (19, 23, 31 bits: B = 8 is the native layout).  Needs
 *              n_refs < 2^tb - 1; an id outside the table is stored as 2^tb - 1.  The buffer must be
 *              16-byte aligned and readable up to the next multiple of 8 bytes; a chunk boundary
 *              must fall on a multiple of 8 records.  bin3c_io.h: b3c_records_pack packs on the host.
 *   add_pairs_same  records of pairs whose two mates lie on ONE reference (four in five Hi-C pairs): B = 3 or
 *              4 little-endian bytes holding the reference id in bits [0, 8B-1) and the pass flag in the top
 *              bit (n_refs < 2^(8B-1) - 1; an id outside the table is stored as all ones).  Same alignment
 *              rules.  The order of records does not matter to the map, so a producer may hand the same-
 *              reference pairs over in this form and only the others as pair records (bin3c_io.h:
 *              b3c_records_split): 3.4 instead of 5 bytes per pair over PCIe on the bench communities.
 *   reduce     radix sort the keys + run-length reduce; returns sizes to the host:
 *              h_sizes[0] = nnz of the upper triangle incl. diagonal
 *              h_sizes[1] = nnz of the full symmetric matrix
 *              h_sizes[2..4] = accepted, ref_excluded, poor_match (contact_map.py:709-716)
 *              h_sizes[5] = map weight = sum of the symmetric matrix (contact_map.py:834-838)
 *   emit       write the canonical CSR (sorted columns, exact uint32 counts):
 *              symmetric != 0 -> full symmetric matrix as get_coo(symm=True) returns it
 *              (diagonal once, off-diagonals mirrored, Q7); else the upper triangle.
 * ------------------------------------------------------------------------------------ */
int64_t b3c_accum_workspace_bytes(int64_t pair_capacity, int32_t n_seq, int32_t n_refs);
int b3c_accum_begin(void *d_ws, int64_t ws_bytes, int64_t pair_capacity, int32_t n_seq,
                    const int32_t *d_tid2idx, int32_t n_refs, void *stream);
int b3c_accum_reset(void *d_ws, void *stream);
int b3c_accum_add_pairs(void *d_ws, const uint64_t *d_records, int64_t n_records, void *stream);
int b3c_accum_add_pairs_packed(void *d_ws, const void *d_bytes, int64_t n_records, int32_t bytes_per_record,
                               void *stream);
int b3c_accum_add_pairs_same(void *d_ws, const void *d_bytes, int64_t n_records, int32_t bytes_per_record,
                             void *stream);
int b3c_accum_reduce(void *d_ws, int64_t *h_sizes, void *stream);
int b3c_accum_emit_csr(void *d_ws, int symmetric, int64_t *d_indptr, int32_t *d_indices,
                       uint32_t *d_counts, void *stream);

/* ------------------------------------------------------------------------------------
 * Sharded accumulation (multi-GPU, SURVEY.md section 8e; driver: bin3c_b200/dist.py).  Each rank
 * classifies its own chunk of the pair records (begin / add_pairs as above), then:
 *
 *   row_hist      d_rowcnt[r] (uint64[n_seq], zeroed by the caller) += directed keys of row r,
 *                 all-reduced by the driver to cut nnz-balanced row ranges
 *   route         turns every canonical key (i<j) into the directed keys (i,j) and (j,i) and
 *                 buckets them by the rank that owns their row: d_splits (int32[n_ranks+1]) are
 *                 the row-range boundaries; d_out receives the buckets back to back;
 *                 h_counts[0..n_ranks] = bucket offsets (exclusive scan, last = total) followed
 *                 by this rank's accepted / ref_excluded / poor_match counters.
 *                 d_scratch needs 1600 bytes.
 *   reduce_block  after the all-to-all: sort + run-length reduce the directed keys received for
 *                 rows [row_lo, row_hi) (the diagonal counts in the workspace must already be
 *                 all-reduced: b3c_accum_offsets gives their location); h_sizes[0] = nnz of the
 *                 row block of the full symmetric matrix
 *   emit_block    local CSR of the row block: local indptr, global sorted columns, exact counts
 * ------------------------------------------------------------------------------------ */
int b3c_accum_offsets(void *d_ws, int64_t *h_offsets /* [4]: counters, diagonal, keys, capacity */);
int b3c_accum_row_hist(void *d_ws, uint64_t *d_rowcnt, void *stream);
int b3c_accum_route(void *d_ws, const int32_t *d_splits, int32_t n_ranks, uint64_t *d_out,
                    int64_t out_capacity, uint64_t *d_scratch, int64_t *h_counts, void *stream);
int b3c_accum_reduce_block(void *d_ws, const uint64_t *d_keys, int64_t n_keys, int32_t row_lo,
                           int32_t row_hi, int64_t *h_sizes, void *stream);
int b3c_accum_emit_block(void *d_ws, int32_t row_lo, int32_t row_hi, int64_t *d_indptr,
                         int32_t *d_indices, uint32_t *d_counts, void *stream);

/* ------------------------------------------------------------------------------------
 * Row blocks.  The row-wise entry points below take a block of n_local rows whose first row is
 * global row `row_lo`: d_indptr is local (n_local + 1 entries, starting at 0), column indices are
 * global, and per-contig vectors (sites, x, mask, newidx) are indexed globally.  A whole matrix
 * is the block row_lo = 0, n_local = n.  This is what the multi-GPU driver shards on.
 *
 * Filter mask.  max_offdiag (sparse_utils.py:269-281) and the two threshold tests of
 * ContactMap.set_primary_acceptance_mask (contact_map.py:888-905).
 * d_signal has n_local entries; b3c_acceptance_mask works on whole vectors of length n.
 * ------------------------------------------------------------------------------------ */
int b3c_max_offdiag_u32(int32_t n_local, int32_t row_lo, const int64_t *d_indptr,
                        const int32_t *d_indices, const uint32_t *d_counts, uint32_t *d_signal,
                        void *stream);
int b3c_max_offdiag_f64(int32_t n_local, int32_t row_lo, const int64_t *d_indptr,
                        const int32_t *d_indices, const double *d_data, double *d_signal,
                        void *stream);
int b3c_acceptance_mask(int32_t n, const int32_t *d_lengths, const uint32_t *d_signal,
                        int64_t min_len, int64_t min_sig, uint8_t *d_mask, void *stream);

/* ------------------------------------------------------------------------------------
 * Site normalisation.  ContactMap._get_sites + fast_norm_fullseq_bysite
 * (contact_map.py:1103-1108, 100-113): out[e] = count[e] * (1.0 / (s_i * s_j)), zero sites
 * counted as one (Q6).  d_sites is the raw int32 site count per contig (global).
 * ------------------------------------------------------------------------------------ */
int b3c_site_norm(int32_t n_local, int32_t row_lo, const int64_t *d_indptr,
                  const int32_t *d_indices, const uint32_t *d_counts, const int32_t *d_sites,
                  double *d_out, void *stream);
/* same on an already-float matrix, in place (ContactMap._norm_seq called on a float map) */
int b3c_site_norm_f64(int32_t n_local, int32_t row_lo, const int64_t *d_indptr,
                      const int32_t *d_indices, double *d_data, const int32_t *d_sites,
                      void *stream);

/* ------------------------------------------------------------------------------------
 * Knight-Ruiz balancing.  kr_biostochastic (sparse_utils.py:90-224).
 *
 *   b3c_kr_run    computes the scale vector x (float64[n]) of the symmetric CSR matrix;
 *                 zero diagonals are treated as one on the working matrix only (Q2).
 *                 h_info (int64[32]): [0] = n_iter, [1] = zero diagonals patched, [2] = outer
 *                 Newton steps, [3] = SpMV phases executed, [4] = CTAs of the persistent grid,
 *                 [5] = SM cycles of the whole kernel, [6..14] = cycles CTA 0 spent working in
 *                 each phase (init, spmv, fix-up, residual, direction, w, step, update, scalar
 *                 reductions), [15..23] = cycles it waited at the grid barrier after each,
 *                 [24] = column slabs of the SpMV operand (0 = gather form), [25] = entries of the
 *                 SpMV stream including slab padding, [26] = (row, slab) segments, [27] = duration
 *                 of the persistent kernel alone in microseconds (CUDA events on `stream`),
 *                 [28..30] = SpMV cycles of the fastest CTA, the slowest CTA and the mean.
 *                 mode 0 = one persistent cooperative kernel (device-side control flow).
 *   b3c_kr_scale  out[e] = x_i * (a_ij * x_j), the entries of X.T.dot(orig.dot(X))
 *                 (sparse_utils.py:223-224, Q9) on the ORIGINAL matrix.
 *   b3c_spmv      y = A.u with the same kernel KR uses (microbench, config C5).
 * ------------------------------------------------------------------------------------ */
/* Tuning / test hooks.  KR's SpMV gathers its operand vector from shared memory, one column slab at
 * a time (see csrc/kr.cu); B3C_OPT_KR_SLAB_WIDTH caps the slab width (default 28672 columns, the most
 * that fits in a CTA's shared memory), B3C_OPT_KR_MAX_SLABS the slab count (default 16, at most 48; wider
 * matrices, or 0, select the form that gathers through L1/L2 -- except that at the default, matrices of up
 * to 48 slabs whose (row, slab) cells hold 6 or more entries on average -- 4 for the packed count stream -- stay in the
 * slab form; b3c_kr_run_peer* applies that rule to its own row block, counting the block's rows rounded up to whole
 * 1024-row chunks, as the stream lays its cells out: a tail block of fewer rows takes the form a 1024-row block with the
 * same entries takes, which b3c_krp_workspace_bytes has room for).  Results are
 * identical up to fp64 summation order.  Workspace sizes depend on these, so set them before the *_workspace_bytes() query.
 * B3C_OPT_KR_FLAGS (default 22) is a bit set for A/B measurements: 1 = order every lane's run of the
 * stream by shared-memory bank (off: the pass costs more than it saves below ~180 SpMV per solve), 2 = align the SpMV CTA ranges with the slabs, 4 = single-word grid
 * barrier (release-add + acquire-poll), 8 = on one GPU the phases that only produce reduction partials
 * hand them over as flagged 8-byte words instead of passing a grid barrier (off: measured slower), 16 = in
 * peer mode (several GPUs) the p.w partials after the `w` phase cross the NVLink as such flagged words
 * instead of a system-fenced flag barrier, 32 / 64 = L2 prefetch of the stream 6 / + 12 chunks ahead (off: no gain
 * measured), 128 = the stream builder orders every 8-entry piece by shared-memory bank pair and rotates it by the lane
 * that will process it, so that the lanes of a half-warp gather from different banks (slab form; off: with shuffled contig
 * order the columns of a piece are random, the order removes 5 % of the gather's wavefronts and its ranking costs the
 * stream builder more than the kernel gains).
 * B3C_OPT_PEER_TIMEOUT_MS (default 60000): how long a cross-GPU flag wait (peer barriers of the sharded
 * accumulation, hand-overs of peer-mode KR) may last before it gives up.  A time-out is reported as
 * B3C_ERR_CUDA by the next call that synchronises and the results of that run are invalid; it is cleared
 * at the start of the next run.
 * B3C_OPT_KR_COUNT_STREAM (default 2): b3c_kr_run_counts / b3c_kr_run_peer_counts stream the raw counts and factor
 * the site normalisation out of the row sums, (A u)_i = (1/s_i) sum_j c_ij (u_j / s_j).  1: uint32 counts, 6 bytes
 * per entry with the 16-bit column.  2 (slab form): packed entries, 16-bit count | 16-bit column = 4 bytes; the high
 * part of a DIAGONAL count above 65535 (intra-contig pairs of a long contig) is applied as a per-row term, and a matrix
 * with an OFF-diagonal count above 65535 falls back to form 1 (detected while the stream is laid out).  0 streams fp64
 * values c_ij / (s_i s_j) (10 bytes per entry), bit-identical to the staged form.  h_info[31] reports the bytes per entry.
 * B3C_OPT_USE_GRAPHS (default 1): the sort-reduce sequences of an accumulator (~60 launches with fixed grids;
 * all sizes are read from device counters) are captured once per workspace as a CUDA graph and replayed. */
enum { B3C_OPT_KR_SLAB_WIDTH = 1, B3C_OPT_KR_MAX_SLABS = 2, B3C_OPT_KR_FLAGS = 3, B3C_OPT_PEER_TIMEOUT_MS = 4,
       B3C_OPT_KR_COUNT_STREAM = 5, B3C_OPT_USE_GRAPHS = 6 };
int b3c_set_option(int32_t key, int64_t value);
/* b3c_accum_plan: the code paths an accumulator of these sizes takes (host-only, no CUDA call), so tests can
 * assert the branch they were written for.  h_out[10] = key bits b per index, shared-memory diagonal (0/1),
 * rank-table mode of the classify kernel (0 gather, 1 pair table, 2 packed table, 3 two-level table), staging
 * keys per warp, contigs of the partial shared-memory diagonal, passes and digit bits of the key sort
 * (bits [0, 2b)), passes and digit bits of the mirror composite's sort, count bits of the composite. */
int b3c_accum_plan(int64_t pair_capacity, int32_t n_seq, int32_t n_refs, int64_t *h_out);
/* b3c_kr_plan: the SpMV operand layout b3c_kr_run* (rows = n) or b3c_kr_run_peer* (rows = the block's row count)
 * chooses for a matrix of n columns and nnz_local entries under the current options (host-only, no CUDA call).
 * counts != 0: the counts form.  h_out[5] = slabs (0 = gather form), S, slab width W, the stream form requested
 * (0 fp64, 1 32-bit counts, 2 packed counts; the build falls back from 2 to 1 when the side list overflows), and the
 * workspace bytes that layout needs. */
int b3c_kr_plan(int32_t n, int64_t nnz_local, int32_t rows, int32_t counts, int64_t *h_out);
/* b3c_kr_rowsum: builds the operand of rows [row_lo, row_hi) exactly as b3c_kr_run_peer* does ([0, n): as b3c_kr_run*)
 * -- d_data for fp64 values, or d_counts with d_sites for the counts form (d_data null) -- and writes to d_q[row -
 * row_lo] the row sums KR's iteration uses for the local rows, (A v)_r plus the zero-diagonal term, with v = d_v
 * (all n columns) taken as the CG operand u (which = 0) or as x of a residual (which = 1).  Synchronises.
 * h_info[8] = slabs (0 = gather form), S, stream bytes per entry, side-list entries, stream entries incl. padding,
 * segments, zero diagonals of the block, workspace bytes the layout needs. */
int b3c_kr_rowsum(int32_t n, int32_t row_lo, int32_t row_hi, int64_t nnz_local, const int64_t *d_indptr,
                  const int32_t *d_indices, const double *d_data, const uint32_t *d_counts, const int32_t *d_sites,
                  int32_t which, const double *d_v, double *d_q, void *d_ws, int64_t ws_bytes, int64_t *h_info,
                  void *stream);

int64_t b3c_kr_workspace_bytes(int32_t n, int64_t nnz);
int b3c_kr_run(int32_t n, int64_t nnz, const int64_t *d_indptr, const int32_t *d_indices,
               const double *d_data, double tol, double delta, double Delta, int32_t max_iter,
               int32_t mode, double *d_x, void *d_ws, int64_t ws_bytes, int64_t *h_info,
               void *stream);
/* Counts form of b3c_kr_run: the matrix is given as the raw uint32 contact counts plus the int32 site
 * count per contig, and every entry is normalised while the SpMV operand is built --
 * a_ij = count_ij * (1.0 / (s_i * s_j)), bit for bit what b3c_site_norm writes
 * (prepare_seq_map's astype(float) + _norm_seq, contact_map.py:929-933, 110-113) -- so the normalised
 * matrix is never materialised.  Same result, same h_info as b3c_kr_run on b3c_site_norm's output. */
int b3c_kr_run_counts(int32_t n, int64_t nnz, const int64_t *d_indptr, const int32_t *d_indices,
                      const uint32_t *d_counts, const int32_t *d_sites, double tol, double delta,
                      double Delta, int32_t max_iter, double *d_x, void *d_ws, int64_t ws_bytes,
                      int64_t *h_info, void *stream);
int b3c_kr_scale(int32_t n_local, int32_t row_lo, const int64_t *d_indptr,
                 const int32_t *d_indices, const double *d_data, const double *d_x, double *d_out,
                 void *stream);
/* is_hermitian (sparse_utils.py:10-18) without the dense N x N temporary (Q11): counts the
 * entries with |a_ij - a_ji| >= tol (a missing mirror entry counts as zero).  Columns must be
 * sorted within rows.  h_count[0] receives the count (the stream is synchronised). */
int b3c_asymmetry_count(int32_t n, const int64_t *d_indptr, const int32_t *d_indices,
                        const double *d_data, double tol, uint64_t *d_scratch, int64_t *h_count,
                        void *stream);
int b3c_spmv(int32_t n, int64_t nnz, const int64_t *d_indptr, const int32_t *d_indices,
             const double *d_data, const double *d_u, double *d_y, void *d_ws, int64_t ws_bytes,
             int32_t prepared, void *stream);
/* b3c_spmv: prepared = 0 builds the SpMV operand and plan for this matrix in d_ws (and synchronises);
 * prepared != 0 reuses what the last prepared = 0 call on the same d_ws built. */

/* ------------------------------------------------------------------------------------
 * Row-block phase API of KR (multi-GPU driver; SURVEY.md section 8e, bin3c_b200/dist.py).  Each
 * rank owns rows [row_lo, row_hi) (1024-row aligned) of the matrix as a local CSR with global
 * columns, and the matching slices of all vectors.  The arithmetic is that of b3c_kr_run; the
 * driver puts collectives between the phases:
 *
 *     phase INIT | all-reduce u | SPMV | RESID | all-reduce partials | scalar OUTER_FIRST
 *     while state != DONE:
 *       INNER : DIR | all-reduce u | SPMV | W | all-reduce PA,PB | scalar ALPHA |
 *               STEP | all-reduce PC (sum), PMIN..PG2 (min) | scalar DECIDE
 *       UPDATE: UPDATE | all-reduce u | SPMV | RESID | all-reduce PA | scalar OUTER
 *
 * u slices a rank does not own are zero, so a SUM all-reduce assembles the vector exactly; the
 * partial arrays hold the identity (0 / +inf) for chunks a rank does not own.
 * setup returns byte offsets into the workspace: h_offsets[0] = u (float64[n]), [1] = x
 * (float64[n]), [2] = partials (float64[7][n_chunks]: sums PA PB PC, then minima), [3] = n_chunks.
 * b3c_krp_state synchronises and returns state (0 done, 1 inner, 2 update), status, n_iter, k,
 * outer steps, SpMV count, zero diagonals of this block.
 * ------------------------------------------------------------------------------------ */
int64_t b3c_krp_workspace_bytes(int32_t n, int64_t nnz_local);
int b3c_krp_setup(int32_t n, int32_t row_lo, int32_t row_hi, int64_t nnz_local,
                  const int64_t *d_indptr, const int32_t *d_indices, const double *d_data,
                  double tol, double delta, double Delta, int32_t max_iter,
                  void *d_ws, int64_t ws_bytes, int64_t *h_offsets, void *stream);
int b3c_krp_phase(void *d_ws, int32_t phase, void *stream);   /* 0 INIT 1 SPMV 2 RESID 3 DIR 4 W 5 STEP 6 UPDATE */
int b3c_krp_scalar(void *d_ws, int32_t which, void *stream);  /* 0 OUTER_FIRST 1 OUTER 2 ALPHA 3 DECIDE */
int b3c_krp_state(void *d_ws, int64_t *h_state /* [8] */, void *stream);

/* ------------------------------------------------------------------------------------
 * Peer mode of KR (multi-GPU, one process per GPU of ONE node).  Every rank runs the same persistent
 * kernel as b3c_kr_run on its row block; the operand vector u and the fixed-shape partials live in
 * an "exchange buffer" per rank that every other rank maps over NVLink (CUDA IPC), and each rank
 * writes its slice of u and its partials straight into all of them (peer stores).  Cross-GPU
 * barriers are release/acquire flags in the same buffers, so an iteration needs no host round
 * trip and no collective call; results are those of the phase API.
 *
 *   b3c_peer_alloc   cudaMalloc + zero `bytes` on the current device; h_handle64 receives the 64-byte
 *                    IPC handle to hand to the other ranks (e.g. with an all-gather)
 *   b3c_peer_open    map another rank's buffer from its handle (peer access is enabled lazily)
 *   b3c_peer_close / b3c_peer_free   undo open / alloc
 *   b3c_kr_exchange_bytes            size of the exchange buffer for an n x n matrix
 *   b3c_kr_run_peer  as b3c_kr_run on rows [row_lo, row_hi); h_exchange (HOST array of n_ranks DEVICE
 *                    pointers) lists the exchange buffer of every rank as seen from this process,
 *                    its own at [rank].  All ranks must call it together (the kernels wait for each
 *                    other); a missing rank ends in B3C_ERR_CUDA after a time-out instead of a hang.
 *                    d_x receives the whole workspace vector x: only rows [row_lo, row_hi) are
 *                    meaningful.  h_info as b3c_kr_run; [27] = microseconds of the persistent kernel.
 * ------------------------------------------------------------------------------------ */
int b3c_peer_alloc(int64_t bytes, void **d_ptr, uint8_t *h_handle64);
int b3c_peer_open(const uint8_t *h_handle64, void **d_ptr);
int b3c_peer_close(void *d_ptr);
int b3c_peer_free(void *d_ptr);
int64_t b3c_kr_exchange_bytes(int32_t n);
int b3c_kr_run_peer(int32_t n, int32_t row_lo, int32_t row_hi, int64_t nnz_local,
                    const int64_t *d_indptr, const int32_t *d_indices, const double *d_data,
                    double tol, double delta, double Delta, int32_t max_iter, int32_t rank,
                    int32_t n_ranks, void *const *h_exchange, double *d_x, void *d_ws,
                    int64_t ws_bytes, int64_t *h_info, void *stream);

/* counts form of b3c_kr_run_peer (see b3c_kr_run_counts) */
int b3c_kr_run_peer_counts(int32_t n, int32_t row_lo, int32_t row_hi, int64_t nnz_local,
                           const int64_t *d_indptr, const int32_t *d_indices,
                           const uint32_t *d_counts, const int32_t *d_sites, double tol,
                           double delta, double Delta, int32_t max_iter, int32_t rank,
                           int32_t n_ranks, void *const *h_exchange, double *d_x, void *d_ws,
                           int64_t ws_bytes, int64_t *h_info, void *stream);

/* ------------------------------------------------------------------------------------
 * Peer exchange arena: the sharded accumulation without a collective library in the data path
 * (SURVEY.md section 8e; the reference has no multi-process form -- this is the partitioned
 * equivalent of Sparse2DAccumulator.get_coo, sparse_utils.py:246-266, one row block per GPU).
 * Every rank allocates one arena (b3c_peer_alloc, b3c_xa_bytes) and maps the others' (b3c_peer_open);
 * h_arena is the HOST array of n_ranks DEVICE pointers as seen from this process, its own at [rank].
 * All calls only enqueue work on `stream` unless stated.  `epoch` is a counter the callers advance
 * together: every barrier / all-reduce call of a rank uses the next value (1, 2, 3, ...).
 *
 *   b3c_peer_barrier        flag barrier between the ranks' streams: work enqueued after it starts
 *                           once every rank has completed what it enqueued before it
 *   b3c_peer_put            copy bytes from d_src into EVERY rank's arena at `offset` (peer stores)
 *   b3c_peer_allreduce_f64  in-place all-reduce of count <= 8 doubles (op 0 = sum, 1 = max), slots
 *                           reduced in rank order: one kernel = put + barrier + reduce
 *   b3c_xa_offsets          h_offsets[0] = mask (uint8[n_seq]), [1] = x (float64[n_seq]), [2] = key
 *                           receive buffer, [3] = diagonal histogram: regions callers put into / view
 *
 *   Sharded accumulation, after b3c_accum_add_pairs on every rank's own records:
 *     b3c_shard_publish       1024-row chunk weights of the local keys, the pair counters and the local
 *                             diagonal histogram into the arenas; resets this rank's receive cursor
 *     (barrier)
 *     b3c_shard_scatter       d_splits (int32[n_ranks+1], device) = row ranges of about equal weight, cut
 *                             at chunk boundaries, identical on every rank; then every canonical key
 *                             (i<j) is written as (i,j) and (j,i) straight into the receive buffer of
 *                             the rank owning its row (one system-scope atomic per owner and tile
 *                             reserves the range; owner-contiguous coalesced peer stores)
 *     (barrier)
 *     b3c_shard_reduce_block  sort + run-length reduce what was received, gather the diagonal counts
 *                             of the own rows from all ranks, build the row pointers; synchronises.
 *                             h_sizes (int64[24]): [0] = entries of this rank's block, [1] = row_lo,
 *                             [2] = row_hi, [3..5] = accepted / ref_excluded / poor_match summed over
 *                             ranks, [6] = directed keys received, [8..8+n_ranks] = the splits.
 *                             Follow with b3c_accum_emit_block(row_lo, row_hi).
 * Counts are integer sums, so the block is bit-identical whatever the number of ranks.
 * ------------------------------------------------------------------------------------ */
int64_t b3c_xa_bytes(int32_t n_seq, int64_t key_capacity);
int b3c_xa_offsets(int32_t n_seq, int64_t key_capacity, int64_t *h_offsets /* [4] */);
int b3c_peer_barrier(void *const *h_arena, int32_t rank, int32_t n_ranks, int32_t n_seq,
                     int64_t key_capacity, uint64_t epoch, void *stream);
int b3c_peer_put(void *const *h_arena, int32_t n_ranks, int64_t offset, const void *d_src,
                 int64_t bytes, void *stream);
int b3c_peer_allreduce_f64(void *const *h_arena, int32_t rank, int32_t n_ranks, int32_t n_seq,
                           int64_t key_capacity, uint64_t epoch, int32_t op, double *d_val,
                           int32_t count, void *stream);
int b3c_shard_publish(void *d_ws, void *const *h_arena, int32_t rank, int32_t n_ranks, void *stream);
int b3c_shard_scatter(void *d_ws, void *const *h_arena, int32_t rank, int32_t n_ranks,
                      int32_t *d_splits, void *stream);
int b3c_shard_reduce_block(void *d_ws, void *const *h_arena, int32_t rank, int32_t n_ranks,
                           const int32_t *d_splits, int64_t *h_sizes, void *stream);

/* ------------------------------------------------------------------------------------
 * Compress + edge weighting.  compress (sparse_utils.py:284-314), get_subspace
 * (contact_map.py:966-982) and the edge loop of to_graph (cluster.py:314-321), on a row block
 * (see "Row blocks"); d_mask and d_newidx have n entries.
 *
 *   count   d_newidx[i] = index of contig i among the accepted ones (or -1), over the whole
 *           mask; d_vmax (float64[1]) = largest kept value of this block (the multi-GPU driver
 *           all-reduces it with MAX before fill);
 *           h_out[0] = accepted contigs (whole mask), [1] = entries kept in this block,
 *           [2] = undirected edges of this block (kept entries with u<=v, self-loops
 *           included, Q8)
 *   fill    the edge list (u, v, w) with w = value * scl, scl = 1/d_vmax when scale != 0
 *           (cluster.py:316, maximum over the kept entries incl. the diagonal, Q8); one value
 *           per undirected edge, taken from the upper-triangle entry (Q9); d_scl receives scl.
 *           For a whole matrix (row_lo = 0, n_local = n) the compressed CSR can be written as
 *           well (d_sub_*; NULL to skip).
 * ------------------------------------------------------------------------------------ */
int64_t b3c_compress_workspace_bytes(int32_t n);
int b3c_compress_count(int32_t n, int32_t row_lo, int32_t n_local, const int64_t *d_indptr,
                       const int32_t *d_indices, const double *d_data, const uint8_t *d_mask,
                       int32_t *d_newidx, void *d_ws, int64_t ws_bytes, double *d_vmax,
                       int64_t *h_out, void *stream);
int b3c_compress_fill(int32_t n, int32_t row_lo, int32_t n_local, const int64_t *d_indptr,
                      const int32_t *d_indices, const double *d_data, const uint8_t *d_mask,
                      const int32_t *d_newidx, void *d_ws, const double *d_vmax, int scale,
                      int64_t *d_sub_indptr, int32_t *d_sub_indices, double *d_sub_data,
                      int32_t *d_edge_u, int32_t *d_edge_v, double *d_edge_w, double *d_scl,
                      void *stream);

/* Fused form for the graph hand-off (to_graph with norm=True, bisto=True, cluster.py:301-321): the
 * edge list straight from the raw counts, the site counts and the KR scale vector.  The value of an
 * entry is x_i * ((count_ij * (1.0 / (s_i * s_j))) * x_j) -- exactly what b3c_site_norm followed by
 * b3c_kr_scale would have stored (contact_map.py:110-113, sparse_utils.py:223-224) -- so neither the
 * normalised nor the balanced matrix is written to memory.  Arguments and outputs as
 * b3c_compress_count / b3c_compress_fill (edge list only); b3c_edges_count leaves one packed record
 * per contig (gapless id, site count, x) in d_ws, which b3c_edges_fill gathers from. */
int b3c_edges_count(int32_t n, int32_t row_lo, int32_t n_local, const int64_t *d_indptr,
                    const int32_t *d_indices, const uint32_t *d_counts, const int32_t *d_sites,
                    const double *d_x, const uint8_t *d_mask, int32_t *d_newidx, void *d_ws,
                    int64_t ws_bytes, double *d_vmax, int64_t *h_out, void *stream);
int b3c_edges_fill(int32_t n, int32_t row_lo, int32_t n_local, const int64_t *d_indptr,
                   const int32_t *d_indices, const uint32_t *d_counts, void *d_ws,
                   const double *d_vmax, int scale, int32_t *d_edge_u, int32_t *d_edge_v,
                   double *d_edge_w, double *d_scl, void *stream);

/* ------------------------------------------------------------------------------------
 * Extent (binned) map length normalisation.  ContactMap._norm_extent with mean_selector
 * (contact_map.py:1147-1165, :25-46): out[e] = count[e] / (1e-3 * mean(L_r, L_c)), d_bin_len[b] = length
 * of the sequence bin b belongs to (global bin index); mean_type 0 geometric, 1 harmonic, 2 arithmetic,
 * -1 none (uint32 -> float64 copy).  The compressed / balanced forms of get_extent_map (:1001-1036) are
 * b3c_compress_* with the mask expanded to bins and b3c_kr_run / b3c_kr_scale on the result.
 * ------------------------------------------------------------------------------------ */
int b3c_extent_norm(int32_t n_local, int32_t row_lo, const int64_t *d_indptr, const int32_t *d_indices,
                    const uint32_t *d_counts, const double *d_bin_len, int32_t mean_type, double *d_out,
                    void *stream);

/* ------------------------------------------------------------------------------------
 * Synthetic pair-record stream (bench / test tool -- NOT part of the hot path; the reference has no
 * counterpart).  SURVEY.md section 8(d): the pair streams of the large BASELINE configs (C3: 4 GB,
 * C4: 16 GB of packed records) are generated on the device, per shard, by a counter-based generator:
 * record t is a pure function of (seed, t) and the community tables, so any sub-range is reproducible
 * on any rank and on the host (bin3c_b200/synth.py: StreamV2.host_records is the bit-exact NumPy
 * mirror the CPU oracle is fed from).  Tables are in genome-sorted contig order s: d_cum_w1[N]
 * normalised cumulative end-1 weight, d_cum_len[N+1] cumulative length, d_genome_sorted[N],
 * d_g_start/d_g_end[G] contig range of a genome, d_tid_of_s[N] BAM reference id, d_excl_tids[n_excl]
 * excluded references.  Writes records [first, first + count) of the stream to d_records.
 * ------------------------------------------------------------------------------------ */
int b3c_synth_pairs(const double *d_cum_w1, const double *d_cum_len, const int32_t *d_genome_sorted,
                    const int32_t *d_g_start, const int32_t *d_g_end, const int32_t *d_tid_of_s,
                    const int32_t *d_excl_tids, int32_t n_contigs, int32_t n_genomes, int32_t n_excl,
                    double p_same, double p_genome, double p_pass, double excl_end_frac, uint64_t seed,
                    uint64_t first, int64_t count, uint64_t *d_records, void *stream);

/* ------------------------------------------------------------------------------------
 * BAM decoding (the step before the path, on the device; bin3c_b200/csrc/bamdec.cu).  A name-sorted
 * BAM file -> the packed pair records of the contig map, the same values in the same order as the host
 * reader (include/bin3c_io.h: b3c_bam_read_pairs) writes, and the same counters.  The host parses the
 * header (b3c_bam_open, b3c_bam_data_offset), reads the file in SLABS of whole BGZF blocks and lists each
 * slab's blocks (b3c_bgzf_scan); the decoder inflates, checks ISIZE and CRC-32, finds the record
 * boundaries, parses and pairs on the device.
 *
 *   workspace_bytes  decoder state, the tid -> index table and per-block scratch for up to max_blocks
 *              blocks per slab
 *   begin      once per file: matcher and insert filter as b3c_bam_set_filter (d_tid2idx: int32[n_refs],
 *              device, may be NULL when min_insert <= 0; copied), data_offset = b3c_bam_data_offset
 *   slab       one slab: d_comp = the slab's compressed bytes (device); d_blocks = int64[3 n_blocks]:
 *              offset of the block in d_comp, BSIZE | ISIZE << 32, offset of the block's first inflated
 *              byte from the slab's first (the exclusive sum of ISIZE); stream_offset = uncompressed stream
 *              offset of the slab's first inflated byte (header blocks included); u_bytes = sum of ISIZE.
 *              The previous slab may end inside a record: h_result[1] of the previous call is the stream
 *              offset where that record starts, and the carry_bytes = stream_offset - h_result[1] bytes
 *              before stream_offset (from the previous call's d_u) are passed as d_carry.  d_u receives the
 *              carry and the inflated blocks (u_capacity >= carry_bytes + u_bytes); it must not overlap
 *              d_carry.  Records go to d_out[0 .. h_result[0]); out_capacity >= (carry_bytes + u_bytes) / 72
 *              + 2 always suffices.  `last` != 0 on the slab that ends the file.  Synchronises the stream
 *              once.  h_result[4]: records written, stream offset of the first record not decoded,
 *              blocks whose record boundary was repaired, informative records.  A malformed file ->
 *              B3C_ERR_FORMAT; b3c_last_error() names the first error and its uncompressed stream offset.
 *   stats      h_stats[0..7] = b3c_bam_stats indices 0-7 (synchronises)
 * ------------------------------------------------------------------------------------ */
int64_t b3c_bamdec_workspace_bytes(int32_t max_blocks, int32_t n_refs);
int b3c_bamdec_begin(void *d_ws, int64_t ws_bytes, int32_t min_mapq, int32_t strong, int32_t min_insert,
                     const int32_t *d_tid2idx, int32_t n_refs, int64_t data_offset, void *stream);
int b3c_bamdec_slab(void *d_ws, const uint8_t *d_comp, const int64_t *d_blocks, int32_t n_blocks,
                    int64_t stream_offset, int64_t u_bytes, const uint8_t *d_carry, int64_t carry_bytes,
                    uint8_t *d_u, int64_t u_capacity, int32_t last, uint64_t *d_out, int64_t out_capacity,
                    int64_t *h_result, void *stream);
int b3c_bamdec_stats(const void *d_ws, int64_t *h_stats, int32_t n_stats, void *stream);

/* ------------------------------------------------------------------------------------
 * Restriction-site counts of a FASTA file (the other input of ContactMap's FASTA path, on the device;
 * bin3c_b200/csrc/sites.cu, sites.cuh).  Per sequence: its length, its site count (or the head and tail
 * site counts of a tip-based map) and the byte range of its name in a NAME ARENA: what
 * seq_sites.fasta_site_table computes from the file read in text mode.  The host reads (and inflates) the
 * file into slabs of up to slab_bytes bytes, cut anywhere; the device does everything else.
 *
 *   workspace_bytes  state, per-slab scratch for slabs of up to slab_bytes (<= B3C_SITES_MAX_SLAB) bytes,
 *              and the saved first and last tip_size bases of the open sequence (tip_size 0: no tips)
 *   begin      once per file: n_patterns distinct patterns (<= B3C_SITES_MAX_PATTERNS), pattern p =
 *              h_lengths[p] (1..B3C_SITES_MAX_LEN) IUPAC masks (A 1, C 2, G 4, T 8, OR-ed) at
 *              h_masks[p * B3C_SITES_MAX_LEN + i], counted h_weights[p] times; host arrays.  Synchronises.
 *   slab       the next n_bytes (>= 1) bytes of the file at d_bytes (device).  d_seqs = int64[seq_capacity][5]
 *              per-sequence table, d_names = the name arena (uint8[names_capacity]); both are kept from slab
 *              to slab and may be moved to a larger allocation between calls (contents copied).  When they
 *              are too small the call writes nothing, returns B3C_ERR_CAPACITY with h_result[0] = rows and
 *              h_result[1] = name bytes needed, and the same slab is passed again.  A byte >= 0x80 in a
 *              line that is not a header -> B3C_ERR_FORMAT (text-mode lengths count characters).
 *              h_result[3]: sequences, name bytes, kept bases so far.  Synchronises the stream once.
 *   finish     after the last slab: d_out = int64[out_rows][5] (out_rows >= sequences): per sequence its
 *              length, name range [lo, hi) in the arena, sites (tip maps: head sites), tail sites (tip maps;
 *              else 0).  h_result[3] as for slab.  Synchronises.
 * ------------------------------------------------------------------------------------ */
#define B3C_SITES_MAX_LEN 16
#define B3C_SITES_MAX_PATTERNS 64
#define B3C_SITES_MAX_SLAB (1LL << 30)
int64_t b3c_sites_workspace_bytes(int64_t slab_bytes, int32_t tip_size);
int b3c_sites_begin(void *d_ws, int64_t ws_bytes, int64_t slab_bytes, const uint8_t *h_masks,
                    const int32_t *h_lengths, const int32_t *h_weights, int32_t n_patterns, int32_t tip_size,
                    void *stream);
int b3c_sites_slab(void *d_ws, const uint8_t *d_bytes, int64_t n_bytes, int64_t *d_seqs, int64_t seq_capacity,
                   uint8_t *d_names, int64_t names_capacity, int64_t *h_result, void *stream);
int b3c_sites_finish(void *d_ws, int64_t *d_seqs, int64_t *d_out, int64_t out_rows, int64_t *h_result,
                     void *stream);

/* ------------------------------------------------------------------------------------
 * The cm_graph.edges text of device edge arrays (bin3c_b200/csrc/edgefmt.cu, edgefmt.cuh): one line
 * "u<sep>v<sep>weight\n" per edge, byte for byte what b3c_edges_write_fmt (include/bin3c_io.h) writes for
 * the same host arrays.  float_style is B3C_FLOAT_REPR or B3C_FLOAT_STR12 of include/bin3c_io.h; sep is
 * any byte (0..255).  A line takes at most B3C_EDGES_MAX_LINE_BYTES bytes (two 11-byte ids, two
 * separators, the 24-byte "-d.dddddddddddddddde-308" and the newline).
 *
 *   workspace_bytes  scratch for calls of up to max_edges edges
 *   text       d_u, d_v (int32) and d_w (float64) hold n_edges edges (device; may be NULL when
 *              n_edges == 0); the text goes to d_text[0 .. *h_bytes) (device, any alignment: the
 *              kernel stores 16-byte words only at 16-byte aligned addresses, and no byte outside
 *              that range is written), text_capacity >= B3C_EDGES_MAX_LINE_BYTES * n_edges.
 *              Synchronises the stream once.
 * ------------------------------------------------------------------------------------ */
#define B3C_EDGES_MAX_LINE_BYTES 49
int64_t b3c_edges_text_workspace_bytes(int64_t max_edges);
int b3c_edges_text(void *d_ws, int64_t ws_bytes, const int32_t *d_u, const int32_t *d_v, const double *d_w,
                   int64_t n_edges, int32_t sep, int32_t float_style, uint8_t *d_text, int64_t text_capacity,
                   int64_t *h_bytes, void *stream);

/* ------------------------------------------------------------------------------------
 * BGZF-framed gzip of a byte stream and back (bin3c_b200/csrc/bgzf.cu, deflate.cuh): the stage hand-off
 * file contact_map.p.gz of io_utils.save_object / load_object(device=True).  The stream is cut into
 * MEMBERS of B3C_BGZF_MEMBER_INPUT bytes (only the last one shorter); each becomes one gzip member with
 * the BGZF header (BC subfield holding BSIZE = member length - 1), one raw-deflate block (dynamic Huffman
 * codes, or stored when that is not longer), CRC-32 and ISIZE.  No member exceeds B3C_BGZF_MEMBER_MAX
 * bytes.  A member is a function of its input bytes only: the output does not depend on how a stream is
 * split into calls, as long as each call but the last passes a multiple of B3C_BGZF_MEMBER_INPUT bytes.
 * Any gzip reader reads the members; the 28-byte BGZF end-of-file member is the caller's to append.
 *
 *   deflate_workspace_bytes  scratch for calls of up to max_members members
 *   deflate    d_in[0 .. n_bytes) (device) -> whole members at d_out[0 .. *h_out_bytes) (device, any
 *              alignment), out_capacity >= B3C_BGZF_MEMBER_MAX * members.  Synchronises the stream once.
 *   inflate    d_comp = whole members (device), d_blocks = int64[3 n_blocks] as b3c_bamdec_slab takes
 *              it (offset in d_comp, BSIZE | ISIZE << 32, offset of the member's inflated bytes in d_out;
 *              b3c_bgzf_scan of include/bin3c_io.h lists them).  Each member is inflated and its ISIZE
 *              and CRC-32 checked; a mismatch -> B3C_ERR_FORMAT, b3c_last_error() naming the first bad
 *              member's uncompressed offset.  d_ws: 8 bytes of device scratch.  Synchronises once.
 * ------------------------------------------------------------------------------------ */
#define B3C_BGZF_MEMBER_INPUT 65280
#define B3C_BGZF_MEMBER_MAX 65536
int64_t b3c_bgzf_deflate_workspace_bytes(int64_t max_members);
int b3c_bgzf_deflate(void *d_ws, int64_t ws_bytes, const uint8_t *d_in, int64_t n_bytes, uint8_t *d_out,
                     int64_t out_capacity, int64_t *h_out_bytes, void *stream);
int b3c_bgzf_inflate(void *d_ws, int64_t ws_bytes, const uint8_t *d_comp, const int64_t *d_blocks,
                     int32_t n_blocks, uint8_t *d_out, int64_t out_capacity, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BIN3C_B200_H */
