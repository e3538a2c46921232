/*
 * bin3c_io -- host-side C ABI of the two steps either side of the contact-map hot path
 * (SURVEY.md section 8f, ranks 1 and 2).  Built as bin3c_b200/libbin3c_io.so (g++ + zlib +
 * pthreads; no CUDA, no htslib).  The device path itself is include/bin3c_b200.h.
 *
 *   b3c_bam_*         name-sorted BAM -> reference table + packed pair records.  Replaces the
 *                     pysam side of the reference: AlignmentFile / header checks
 *                     (contact_map.py:534-545), next_informative (:624-629), the pairing loop
 *                     (:720-731), the matchers (:612-622) and the min_insert filter (:761-766).
 *                     BGZF blocks are inflated on a pool of threads, two batches ahead of the
 *                     parser; the parser is the reference's sequential state machine.
 *   b3c_edges_write   edge arrays -> the text file nx.write_edgelist(g, path, data=['weight'],
 *                     delimiter=' ') produces (cluster.py:139-151): one "u v weight" line per
 *                     undirected edge, weight printed as Python's str(float) prints it (Python 3: the
 *                     shortest round-trip decimal; Python 2.7: 12 significant digits).  Formatted on a
 *                     pool of threads.
 *
 * All pointers are HOST pointers.  Functions return 0 (or a non-negative count) on success and a
 * negative b3c_io_status on failure; b3c_io_last_error() returns a thread-local message.
 *
 * Packed pair record (uint64, little endian), identical to include/bin3c_b200.h:
 *     bits  0..30  BAM reference id of the first record of the pair   (r1.reference_id)
 *     bit   31     pass flag: both mates satisfy the matcher          (contact_map.py:737)
 *     bits 32..62  BAM reference id of the second record              (r2.reference_id)
 *     bit   63     0
 * A reference id outside [0, n_refs) is stored as 0x7fffffff (never in the index table, so the
 * pair is counted ref_excluded like `r.reference_id not in _idx`, contact_map.py:733).
 */
#ifndef BIN3C_IO_H
#define BIN3C_IO_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    B3C_IO_OK = 0,
    B3C_IO_ERR_ARG = -1,      /* bad argument                                                   */
    B3C_IO_ERR_OPEN = -2,     /* file cannot be opened / written                                */
    B3C_IO_ERR_FORMAT = -3,   /* not BGZF / not BAM / truncated / CRC mismatch                   */
    B3C_IO_ERR_SORT = -4      /* @HD SO is not 'queryname' (IOError, contact_map.py:537-538)     */
} b3c_io_status;

int b3c_io_version(void);
const char *b3c_io_last_error(void);

typedef struct b3c_bam b3c_bam;

/* Open a BAM file and parse its header (magic, SAM text, reference table).  n_threads <= 0: one
 * inflate thread per online core.  require_queryname != 0 enforces contact_map.py:537-538. */
int b3c_bam_open(const char *path, int32_t n_threads, int32_t require_queryname, b3c_bam **out);
void b3c_bam_close(b3c_bam *bam);

/* header: bam.references / bam.lengths (contact_map.py:545) and the raw SAM text */
int32_t b3c_bam_n_refs(const b3c_bam *bam);
const char *b3c_bam_ref_name(const b3c_bam *bam, int32_t tid);
int64_t b3c_bam_ref_lengths(const b3c_bam *bam, int64_t *h_lengths, int32_t capacity);
int64_t b3c_bam_header_text(const b3c_bam *bam, char *h_text, int64_t capacity);   /* returns the full length */

/* Uncompressed stream offset of the first alignment record (the end of the header parsed by b3c_bam_open). */
int64_t b3c_bam_data_offset(const b3c_bam *bam);

/* The BGZF block table of a host buffer that starts at a block: for each complete block, its offset in the buffer,
 * BSIZE (the block's length minus one, from the BC extra subfield) and ISIZE (from the trailer).  Stops at `capacity`
 * blocks or at the first block the buffer does not hold completely; *h_consumed = the bytes of the blocks listed (the
 * next block starts there).  The header checks are those of the reader (gzip magic, the BC subfield, ISIZE <= 64 KiB)
 * and fail with B3C_IO_ERR_FORMAT; a block cut off by the end of the buffer fails the same way when at_eof != 0 (the
 * file ends there), and ends the scan otherwise.  Returns the number of blocks listed or a negative status. */
int64_t b3c_bgzf_scan(const uint8_t *h_buf, int64_t n_bytes, int32_t at_eof, int64_t *h_offsets, int32_t *h_bsize,
                      int32_t *h_isize, int64_t capacity, int64_t *h_consumed);

/* Matcher and insert filter; call before the first read.
 *   min_mapq     r.mapping_quality >= min_mapq                         (_simple_match, :612-613)
 *   strong       > 0: also the 5'-end CIGAR op must be M with length >= strong; a record without
 *                CIGAR fails                                           (_strong_match, :615-619)
 *   min_insert   > 0 (needs h_tid2idx): a pair that passes the exclusion and matcher tests, whose
 *                read-1 mate is flagged proper-pair and has r2.pos - r1.pos < min_insert, is
 *                dropped here and counted short_insert                 (:744-745, :761-766)
 *   h_tid2idx    BAM reference id -> internal index or -1 (make_reverse_index('refid'), :703);
 *                copied; may be NULL when min_insert == 0 */
int b3c_bam_set_filter(b3c_bam *bam, int32_t min_mapq, int32_t strong, int32_t min_insert,
                       const int32_t *h_tid2idx, int32_t n_refs);

/* Decode until `capacity` records are written or the file ends.  Returns the number of records
 * written (0 = end of file) or a negative status.  Consecutive calls continue the stream. */
int64_t b3c_bam_read_pairs(b3c_bam *bam, uint64_t *h_records, int64_t capacity);

/* The binned EXTENT map (contact_map.py:779-788; bins from ExtentGrouping, :116-156).  After b3c_bam_set_extent the
 * 5'-end position of every record is tracked (r.pos, or r.pos + r.alen for a reverse read, :757-758) and
 * b3c_bam_read_pairs_extent writes, beside each pair record, an EXTENT record of the same layout with global bin
 * numbers in place of reference ids: find_nearest (:49-62) of the position among the upper bin edges of the mate's
 * sequence.  A mate on a reference outside the index table gets 0x7fffffff.  Fed to an accumulator over total_bins
 * bins with the identity index table, the extent records give the extent map and the same three counters.
 *   h_tid2idx       BAM reference id -> sequence index or -1, all n_refs references
 *   h_first_bin     [n_seq] global number of the first bin of a sequence
 *   h_edge_ptr      [n_seq + 1] offsets into h_upper_edges; h_upper_edges[h_edge_ptr[i] .. h_edge_ptr[i+1]) are the
 *                   ascending upper edges of the bins of sequence i (edges[1:] of ExtentGrouping) */
int b3c_bam_set_extent(b3c_bam *bam, const int32_t *h_tid2idx, int32_t n_refs, const int64_t *h_first_bin,
                       const int64_t *h_edge_ptr, const int64_t *h_upper_edges, int32_t n_seq);
int64_t b3c_bam_read_pairs_extent(b3c_bam *bam, uint64_t *h_records, uint64_t *h_extent_records, int64_t capacity);

/* The TIP-BASED map (contact_map.py:631-670, 791-798; the N x N x 2 x 2 tensor of sparse_utils.py:317-409).  After
 * b3c_bam_set_tips every pair that passes the exclusion and matcher tests (and the insert filter) is assigned the
 * sequence end each mate's 5' position falls in -- ends of tip_size bp, or the nearer end of a sequence of at most
 * 2 tip_size bp -- and b3c_bam_read_pairs_tips writes its record with the DOUBLED ids 2 * tid + tip (0 = head,
 * 1 = tail); a pair with a mate in neither end is dropped and counted not_tip (b3c_bam_stats, index 8).  Fed to an
 * accumulator over 2 N ids (table entry 2 t + k -> 2 idx[t] + k), the records give the flattened, symmetric
 * 2N x 2N tensor.  On ONE sequence the reference keeps [tip(read 1), tip(read 2)] unordered (no swap for ix1 == ix2,
 * :774-777): h_tip10[i] = 1 marks the accepted (tail, head) pairs, which the symmetric accumulator merges with the
 * (head, tail) ones, so that the host can take them apart again.  Does not combine with extent records. */
int b3c_bam_set_tips(b3c_bam *bam, int64_t tip_size, const int32_t *h_tid2idx, int32_t n_refs);
int64_t b3c_bam_read_pairs_tips(b3c_bam *bam, uint64_t *h_records, uint8_t *h_tip10, int64_t capacity);

/* h_stats[0] alignments read (what bam.count(until_eof=True) returns once the file is exhausted)
 * h_stats[1] informative alignments (mapped, primary, not supplementary; :628)
 * h_stats[2] pairs found (records written + short_insert + not_tip)
 * h_stats[3] short_insert (:765)
 * h_stats[4] informative alignments left without a mate
 * h_stats[5] BGZF blocks inflated
 * h_stats[6] compressed bytes consumed
 * h_stats[7] uncompressed bytes produced
 * h_stats[8] not_tip (:792-794; tip records only) */
int b3c_bam_stats(const b3c_bam *bam, int64_t *h_stats, int32_t n_stats);

/* Narrow pair records for the host->device copy (include/bin3c_b200.h: b3c_accum_add_pairs_packed).
 * b3c_records_bytes: the smallest of 5, 6, 8 bytes per record that holds reference ids of a table of n_refs.
 * b3c_records_pack: n native records -> n * bytes_per_record bytes (h_out sized to the next multiple of 8 bytes;
 * the tail is zeroed); ids >= 2^tb - 1 (the native out-of-table marker included) become 2^tb - 1.  Returns the
 * number of bytes written (a multiple of 8) or a negative status.  b3c_records_unpack is the inverse. */
int32_t b3c_records_bytes(int64_t n_refs);
int64_t b3c_records_pack(const uint64_t *h_records, int64_t n, int32_t bytes_per_record, uint8_t *h_out, int32_t n_threads);
int64_t b3c_records_unpack(const uint8_t *h_bytes, int64_t n, int32_t bytes_per_record, uint64_t *h_records);

/* The narrowest hand-over: pairs whose mates lie on ONE reference (four in five Hi-C pairs) need one id, not two.
 * b3c_records_same_bytes: 3 or 4 bytes per same-reference record for a table of n_refs (id in bits [0, 8B-1), pass
 * flag in the top bit; include/bin3c_b200.h: b3c_accum_add_pairs_same).  b3c_records_split: n native records -> the
 * same-reference ones as such records into h_out_same, the others as bytes_per_record-byte pair records into
 * h_out_pair, each in input order, each buffer sized to the next multiple of 8 bytes (tail zeroed);
 * h_counts[0] = same-reference records, h_counts[1] = pair records.  With both output pointers NULL only the counts
 * are produced.  Returns n or a negative status.  (The contact map does not depend on the order of its records.) */
int32_t b3c_records_same_bytes(int64_t n_refs);
int64_t b3c_records_split(const uint64_t *h_records, int64_t n, int32_t bytes_per_record, int32_t bytes_per_same,
                          uint8_t *h_out_same, uint8_t *h_out_pair, int64_t *h_counts, int32_t n_threads);

/* How a weight is printed.  networkx prints it with str(): the shortest round-trip decimal on Python 3
 * (== repr), '%.12g' plus '.0' on integer-looking values on the Python 2.7 the reference pins. */
typedef enum {
    B3C_FLOAT_REPR = 0,       /* Python 3 str(float) / repr(float)                               */
    B3C_FLOAT_STR12 = 1       /* Python 2.7 str(float): 12 significant digits                    */
} b3c_float_style;

/* Write `n_edges` lines "u<sep>v<sep>weight\n" to `path` (truncating).  Returns bytes written.
 * b3c_edges_write prints B3C_FLOAT_REPR. */
int64_t b3c_edges_write(const char *path, const int32_t *h_u, const int32_t *h_v, const double *h_w,
                        int64_t n_edges, char sep, int32_t n_threads);
int64_t b3c_edges_write_fmt(const char *path, const int32_t *h_u, const int32_t *h_v, const double *h_w,
                            int64_t n_edges, char sep, int32_t float_style, int32_t n_threads);
/* Format one weight; returns the length (buffer of >= 32 bytes, NUL terminated). */
int32_t b3c_format_weight(double w, char *h_buf, int32_t capacity);
int32_t b3c_format_weight_fmt(double w, int32_t float_style, char *h_buf, int32_t capacity);

#ifdef __cplusplus
}
#endif
#endif /* BIN3C_IO_H */
