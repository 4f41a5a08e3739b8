/*
 * snacc_b200.h -- C ABI of libsnacc_b200.so: the B200 (sm_100a) replacement for the compressor
 * fan-out of snacc's all-pairs NCD hot path.
 *
 * The reference has no FFI; its seam is the Python call boundary
 *     compressed_size(sequences, algorithm, reverse_complement)   snacc/pairwise_ncd.py:42-90
 * driven N + N*N times by the thread pool in                     snacc/cli.py:104-129
 * and followed by compute_distance()                             snacc/pairwise_ncd.py:93-111
 *                                                                snacc/cli.py:131-136.
 * The entry points below are what a ctypes/cffi binding inside snacc would call instead (the stub
 * is shown in INTEGRATION.md).  Plain pointers and sizes only; no C++ or torch types; functions
 * return 0 on success or a negative snacc_status and never throw or abort.  All *host* buffers are
 * owned by the caller; device memory is owned by the opaque context.
 *
 * Compressed sizes returned here are len(compressed bytes) exactly as the reference's compressor
 * call would produce them (lz4framed.compress / gzip.compress / zlib.compress), WITHOUT the +33
 * sys.getsizeof bias of pairwise_ncd.py:90; snacc_ncd() adds the bias it is given.
 */
#ifndef SNACC_B200_H
#define SNACC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct snacc_ctx snacc_ctx;

enum snacc_status {
    SNACC_OK = 0,
    SNACC_ERR_CUDA = -1,        /* a CUDA runtime call or kernel failed (message in snacc_last_error) */
    SNACC_ERR_ARG = -2,         /* bad argument */
    SNACC_ERR_EMPTY = -3,       /* a sequence is empty (reference raises ValueError, pairwise_ncd.py:37) */
    SNACC_ERR_CODEC = -4,       /* codec not supported on the GPU path (reference: KeyError / other libs) */
    SNACC_ERR_STATE = -5,       /* nothing uploaded yet */
    SNACC_ERR_TOO_LARGE = -6    /* a stream would exceed 2 GiB - 1, or a deflate call cannot fit its x-side state,
                                   working buffers and one y in device memory (message: bytes needed, bytes free) */
};

/* codec ids: which reference compressor call is reproduced */
enum snacc_codec {
    SNACC_LZ4F = 0,    /* lz4framed.compress(b)   pairwise_ncd.py:80  (LZ4 frame, 64 KiB linked blocks) */
    SNACC_GZIP9 = 1,   /* gzip.compress(b)        pairwise_ncd.py:74  (deflate level 9, +18 wrapper)    */
    SNACC_ZLIB6 = 2,   /* zlib.compress(b)        pairwise_ncd.py:78  (deflate level 6, +6 wrapper)     */
    SNACC_BZIP2_9 = 3  /* bz2.compress(b)         pairwise_ncd.py:76  (bzip2 level 9, 900 kB blocks)    */
};

/* NCD formulas for snacc_ncd */
enum snacc_formula {
    SNACC_NCD_REFERENCE = 0,   /* min over both orders, pairwise_ncd.py:106-111 (default, bit-identical CSV) */
    SNACC_NCD_ONE_ORDER = 1    /* (C(xy) - min) / max using S[i][j] only (README "fast mode" semantics)      */
};

int snacc_version(void);                                  /* 10000*major + 100*minor + patch */

/* Host-side helper, no GPU involved (replaces the per-job Bio.SeqIO parse of pairwise_ncd.py:29-36, done ONCE per
 * file): residues of every FASTA record of raw[0..n) -- records start at lines beginning with '>', sequence lines are
 * right-stripped and lose blanks and CRs -- concatenated into out (room for n bytes); rec_len receives the length of
 * the first max_recs records.  Returns the number of records (>= 0) or a negative snacc_status. */
int64_t snacc_fasta_parse(const uint8_t *raw, uint64_t n, uint8_t *out, uint64_t *out_len, uint64_t *rec_len,
                          int64_t max_recs);
/* Host-side helper, no GPU involved (replaces the pandas pivot + to_csv of cli.py:138-142 for matrices too large for a
 * DataFrame of N^2 Python objects): writes `header_line` and then, for r = 0..n-1, the line
 * row_labels[order[r]] , D[order[r]][order[0]] , ... , D[order[r]][order[n-1]]  with every double as Python's repr()
 * prints it (shortest round-trip digits; NaN = empty cell, as to_csv).  Labels arrive already quoted (csv.QUOTE_MINIMAL).
 * `threads` <= 0: all host threads.  Returns SNACC_OK or SNACC_ERR_ARG (bad argument / I/O error). */
int snacc_csv_write(const char *path, const char *header_line, const char *const *row_labels, const double *D, int64_t n,
                    const int32_t *order, int threads);
const char *snacc_last_error(const snacc_ctx *ctx);       /* NUL-terminated, owned by ctx; "" if none */

/* replaces: ThreadPoolExecutor construction, cli.py:104 */
int snacc_ctx_create(int device_id, snacc_ctx **out);
void snacc_ctx_destroy(snacc_ctx *ctx);

/*
 * Upload the corpus once (replaces the 2N^2+N FASTA re-reads of pairwise_ncd.py:29-36).
 *   bytes        concatenation of all sequences, one byte per base, case preserved (host memory)
 *   seq_offsets  n_seqs + 1 offsets into bytes; sequence i = bytes[seq_offsets[i] : seq_offsets[i+1]]
 *   rec_offsets  n_recs + 1 offsets of the FASTA records (every sequence is a whole number of
 *                records); may be NULL when reverse_complement == 0
 *   reverse_complement  non-zero: each record is reverse-complemented ON THE DEVICE
 *                (pairwise_ncd.py:33-34: per record, IUPAC-aware, case-preserving), records stay in
 *                file order
 */
int snacc_upload(snacc_ctx *ctx, const uint8_t *bytes, const uint64_t *seq_offsets, int32_t n_seqs,
                 const uint64_t *rec_offsets, int64_t n_recs, int reverse_complement);

/* Same, but `bytes` is a DEVICE pointer on the context's device (e.g. a tensor that arrived by
 * NCCL broadcast); offsets are host arrays. */
int snacc_upload_device(snacc_ctx *ctx, const void *d_bytes, const uint64_t *seq_offsets, int32_t n_seqs,
                        const uint64_t *rec_offsets, int64_t n_recs, int reverse_complement);

/* Copy sequence i (after the optional on-device reverse complement) back to host; out must hold
 * its length.  Testing / debugging aid. */
int snacc_download_sequence(snacc_ctx *ctx, int32_t i, uint8_t *out);

/* replaces the singles fan-out cli.py:108-116: out[k] = len(compress(seq[idx[k]])) */
int snacc_single_sizes(snacc_ctx *ctx, int codec, const int32_t *idx, int64_t n, int64_t *out);

/* replaces the pairs fan-out cli.py:120-129 for an explicit job list:
 * out[k] = len(compress(seq[xs[k]] + seq[ys[k]])) */
int snacc_pair_sizes(snacc_ctx *ctx, int codec, const int32_t *xs, const int32_t *ys, int64_t n_jobs,
                     int64_t *out);

/* A rectangular tile of the ordered-pair matrix: rows [row0,row0+n_rows) x cols [col0,col0+n_cols),
 * out row-major n_rows*n_cols.  This is the unit a rank owns in the multi-GPU sharding. */
int snacc_tile_sizes(snacc_ctx *ctx, int codec, int32_t row0, int32_t n_rows, int32_t col0, int32_t n_cols,
                     int64_t *out);

/*
 * Multi-GPU (one context per GPU, one process per GPU): for the deflate codecs the per-sequence preparation is the
 * part of a run that does not shrink when the pair jobs are split over ranks, so ranks prepare disjoint bands of the
 * sequences -- snacc_single_sizes on the band does it -- and exchange what a pair stream x.* needs of x (its parse
 * checkpoint and the size of x alone) as opaque fixed-size records: export on the rank that owns x, all-gather (NCCL),
 * import on the others.  A rank then only needs the full preparation of the sequences it uses as y.  The reference
 * has no counterpart (single process, cli.py:104); record_bytes == 0 means the codec has nothing to exchange (LZ4).
 */
int64_t snacc_prefix_record_bytes(const snacc_ctx *ctx, int codec);
int snacc_export_prefix(snacc_ctx *ctx, int codec, const int32_t *seqs, int64_t n, void *out /* n records */);
int snacc_import_prefix(snacc_ctx *ctx, int codec, const int32_t *seqs, int64_t n, const void *in /* n records */);

/* replaces compute_distance (pairwise_ncd.py:93-111) + the loop cli.py:131-136, in float64:
 * D[i*n+j] from C[n], S[n*n] (raw lengths) with `bias` added to every size (33 = sys.getsizeof(b"")). */
int snacc_ncd(snacc_ctx *ctx, const int64_t *C, const int64_t *S, int32_t n, int formula, int32_t bias,
              double *D);

/* Downstream of the matrix (SURVEY.md 8f rank 4): metrify -- 0.5 (D + D^T), zero diagonal, snacc/misc.py:20-25 -- when
 * `metrify` is non-zero, then UPGMA, i.e. scipy.cluster.hierarchy.linkage(squareform(D_sym), method='average') of
 * snacc/distmatrix_to_tree.py:9-15.  Z receives scipy's linkage matrix, (n-1) rows of (id_a < id_b, height, leaves),
 * bit for bit, ties included (scipy's nearest-neighbour chain, stable sort by height and relabelling).  Returns
 * SNACC_ERR_ARG, with a message, for input scipy rejects: n < 2, a non-finite entry in the matrix to be clustered
 * (after metrify), and with `metrify` == 0 an asymmetric matrix or a non-zero diagonal. */
int snacc_upgma(snacc_ctx *ctx, const double *D, int32_t n, int metrify, double *Z);

/* ---- instrumentation used by bench.py ---- */
/* device milliseconds (CUDA events on the library's stream) spent in codec kernels during the last
 * sizes call, and the number of kernel launches it made */
int snacc_last_kernel_ms(const snacc_ctx *ctx, double *ms, int64_t *launches);
/* named statistics of the last sizes call: "main_kernel_ms" (dominant kernel only), "total_kernel_ms",
 * "launches", "packed_jobs", "bytewise_jobs", "deflate_serial_jobs" (pair streams of a deflate call that took
 * the full serial parse after their canonical-stream shortcut met a block that might be stored),
 * "deflate_parallel_prep_seqs" (sequences whose parse alone was done in parallel chunks), "deflate_bands" (y layouts
 * of the last deflate call: 1 when its state fit in device memory at once), "deflate_state_bytes" (peak device bytes of
 * deflate per-sequence state plus working buffers during the last deflate call), "deflate_prepared_seqs" (full
 * preparations -- index, match table, parse alone -- the last deflate call made), "lz4_segments"
 * (segments per tile of the last linked-regime LZ4 pair launch), "bzip2_blocks" (blocks sorted and counted),
 * "bzip2_smem_blocks" (of those, sorted in shared memory), "bzip2_prefix_blocks" (closed blocks of an x taken from an
 * earlier computation instead of being recomputed), "bzip2_rle_gather_ms", "bzip2_bwt_small_ms", "bzip2_bwt_large_ms",
 * "bzip2_bits_ms" (device time of the bzip2 stages: RLE1 + block gather, BWT in shared / global memory, MTF + Huffman
 * table choice + bit count) */
int snacc_get_stat(const snacc_ctx *ctx, const char *name, double *out);
/* tunables: 0 = default.  `streams_in_flight` bounds the number of concurrently parsed streams;
 * `invalidate_caches` (any value) drops every per-sequence precomputation so the next call redoes it;
 * `lz4_packed` 0 forces the byte-wise LZ4 kernels; `deflate_canonical` 0 makes every deflate pair stream take
 * the full serial parse instead of the canonical symbol stream of y; `deflate_junction` 2 computes every junction
 * table without the 6-byte-index shortcut, `deflate_index6` 0 every match table from the 3-byte chain walk
 * `deflate_parallel_prep` 0 parses every sequence alone serially, `deflate_tail_index` 0 builds the whole 3-byte
 * index for x-only sequences, `deflate_band_bytes` b > 0 caps the deflate y-side state of one band at b bytes (0: plan
 * from free device memory), `lz4_segments` k forces k segments per LZ4 tile, `bzip2_smem` 0 sorts every bzip2 block
 * in global memory, `bzip2_prefix` 0 recomputes the closed blocks of x for every job x.y (all for tests: same
 * results). */
int snacc_set_option(snacc_ctx *ctx, const char *name, int64_t value);

#ifdef __cplusplus
}
#endif
#endif
