/* frender_b200 -- C-ABI of the B200-native scan/demux hot path of njspix/frender.
 *
 * The reference (/root/reference/frender.py, "F:" below) is a single Python script
 * with no FFI of its own; the entry points here are what a ctypes binding inside
 * frender.py would call in place of the Python functions named beside each group
 * (INTEGRATION.md shows that binding).  Conventions: every function returns an int
 * status (0 = FRB_OK, <0 = error class), the message of the last error on a
 * context is available from frb_last_error(); the caller owns all host memory, the
 * library owns all device memory; one context per GPU, a context is not
 * thread-safe, distinct contexts may be driven from distinct threads (ctypes
 * releases the GIL); no exceptions cross the ABI; there is no CPU fallback --
 * every compute entry point fails with FRB_ERR_CUDA when no sm_100 device is usable.
 *
 * Packed keys.  An index string ("i7+i5" or "i7") over the alphabet {A,C,G,T,N,+}
 * is stored as 3 bits per symbol, symbol i in bits [3i, 3i+3), 0 terminating:
 *   A=1 C=2 G=3 T=4 N=5 '+'=6 (7 = "other", only ever produced for sample-sheet
 * symbols outside ACGTN, which can never equal a read symbol -- F:226-230).
 * 21 symbols fit (10+1+10).  The map is injective, so counting packed keys equals
 * counting strings (F:172-177).  Anything else in a read's key is a hard error
 * (FRB_ERR_BAD_ALPHABET / FRB_ERR_KEY_TOO_LONG): documented deviation, DESIGN.md.
 *
 * Wide keys.  A context set to 128-bit keys (frb_set_key_width) takes index fields of up
 * to 42 symbols as two words (lo, hi): symbol i < 21 at bits [3i, 3i+3) of lo, symbol
 * 21 <= i < 42 at bits [3(i-21), 3(i-21)+3) of hi, same codes.  A key of <= 21 symbols
 * has hi = 0 and lo = its narrow packing, so a wide context counts, orders and writes
 * such keys exactly as a narrow one.  No real key sets bit 63 of lo (FRB_EMPTY_KEY stays
 * free).  43 symbols or more are FRB_ERR_KEY_TOO_LONG.  On a wide context the narrow
 * calls keep working and take hi = 0; frb_scan_chunk_dev with per-read keys_out,
 * frb_total_merge, frb_allmerge, frb_shardmerge and frb_demux_ok with host file lists
 * return FRB_ERR_STATE.
 */
#ifndef FRENDER_B200_H
#define FRENDER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FRB_OK 0
#define FRB_ERR_CUDA (-1)          /* CUDA runtime / no device                                   */
#define FRB_ERR_ARG (-2)           /* bad argument                                               */
#define FRB_ERR_BAD_HEADER (-3)    /* header line without a 2nd space token (IndexError, F:169)  */
#define FRB_ERR_BAD_ALPHABET (-4)  /* key symbol outside ACGTN+                                  */
#define FRB_ERR_KEY_TOO_LONG (-5)  /* key longer than 21 symbols (42 on a wide context)          */
#define FRB_ERR_TABLE_FULL (-6)    /* unique-key table exhausted: recreate with a larger log2    */
#define FRB_ERR_BAD_LENGTH (-7)    /* key/sheet index lengths differ (AssertionError F:227) or a
                                      key has no '+' (ValueError F:306)                          */
#define FRB_ERR_KEY_NOT_FOUND (-8) /* demux: key absent from the results table (F:807-810)       */
#define FRB_ERR_NCCL (-9)
#define FRB_ERR_IO (-10)           /* file / gzip error                                          */
#define FRB_ERR_STATE (-11)        /* call out of sequence                                       */

#define FRB_RULE_SCAN 0            /* 2nd space token, last ':' field (F:169)                    */
#define FRB_RULE_DEMUX 1           /* last ':' field of the whole line (F:778)                   */

#define FRB_GZ_FORMAT_PLAIN 0      /* demux stream: routed bytes as they are                     */
#define FRB_GZ_FORMAT_GZIP 1       /* one gzip member per cell                                   */
#define FRB_GZ_FORMAT_BGZF 2       /* BGZF blocks (htslib / bgzip) per cell                      */

#define FRB_TYPE_UNDETERMINED 0
#define FRB_TYPE_INDEX_HOP 1
#define FRB_TYPE_DEMUXABLE 2
#define FRB_TYPE_AMBIGUOUS 3

#define FRB_EMPTY_KEY 0xFFFFFFFFFFFFFFFFull
#define FRB_CARRY 0xFFFFFFFFFFFFFFFFull /* line_base: continue from the previous chunk         */

typedef struct frb_ctx frb_ctx;

/* ---- library / context ------------------------------------------------------------------ */
int frb_version(void);
int frb_device_count(int* n);
/* table_log2: log2 of the slot count of the per-file and total unique-key tables (32 B/slot). */
int frb_create(int device, uint32_t table_log2, frb_ctx** out);
void frb_destroy(frb_ctx* ctx);
const char* frb_last_error(frb_ctx* ctx); /* ctx may be NULL: last error of a failed create     */
int frb_sync(frb_ctx* ctx);               /* wait for all queued work, surface device errors    */

/* ---- memory helpers ------------------------------------------------------------------------ */
int frb_host_alloc(void** p, size_t nbytes); /* pinned */
int frb_host_free(void* p);
int frb_dev_alloc(frb_ctx* ctx, size_t nbytes, void** dptr);
int frb_dev_free(frb_ctx* ctx, void* dptr);
int frb_h2d(frb_ctx* ctx, void* dptr, const void* host, size_t nbytes); /* synchronous         */
int frb_d2h(frb_ctx* ctx, void* host, const void* dptr, size_t nbytes); /* synchronous         */
int frb_mem_info(frb_ctx* ctx, uint64_t* free_bytes, uint64_t* total_bytes);

/* ---- key packing (host side, exact inverse pair) ------------------------------------------- */
/* Scan-results CSV, one row per unique key in the order given (F:499-501: csv.DictWriter, default dialect;
 * idx1,idx2,matched_idx1,matched_idx2,read_type,sample_name,reads,demux_ok).  m1/m2/sample_row index the
 * string tables of the sheet (-1 = empty field).  Host-only: no context, no device work.                 */
int frb_write_scan_csv(const char* path, const uint64_t* keys, const uint64_t* counts, const int32_t* m1,
                       const int32_t* m2, const uint8_t* read_type, const int32_t* sample_row,
                       const uint8_t* demux_ok, uint64_t n, const char* const* idx1_strings,
                       const char* const* idx2_strings, const char* const* id_strings, uint32_t rows,
                       int single_index);
int frb_pack_key(const char* s, size_t len, int sheet_mode, uint64_t* out);
int frb_unpack_key(uint64_t key, char* out23); /* writes <= 21 chars + NUL, returns length       */
/* wide keys: (lo, hi), up to 42 symbols; frb_unpack_key2 writes <= 42 chars + NUL, returns length */
int frb_pack_key2(const char* s, size_t len, int sheet_mode, uint64_t* lo, uint64_t* hi);
int frb_unpack_key2(uint64_t lo, uint64_t hi, char* out44);
/* frb_write_scan_csv with the upper words of wide keys (keys_hi NULL: all zero) */
int frb_write_scan_csv2(const char* path, const uint64_t* keys, const uint64_t* keys_hi, const uint64_t* counts,
                        const int32_t* m1, const int32_t* m2, const uint8_t* read_type, const int32_t* sample_row,
                        const uint8_t* demux_ok, uint64_t n, const char* const* idx1_strings,
                        const char* const* idx2_strings, const char* const* id_strings, uint32_t rows,
                        int single_index);

/* ---- hot path A: read-name parse + unique-combination counter ------------------------------
 * Replaces scan_file F:154-181 and tally_barcodes F:183-207.
 *   frb_scan_begin      one input file starts: clears the per-file table; `file_ordinal` is
 *                       the position in the file list (first-appearance order of "total",
 *                       F:199-205); read_limit = -s head sample (0 = none, F:163-165).
 *   frb_scan_chunk_*    feed decompressed FASTQ bytes.  A chunk must begin at the start of a
 *                       line.  line_base = number of lines of this file before the chunk, or
 *                       FRB_CARRY to continue counting from the previous chunk of the file.
 *                       _host: pinned or pageable host memory, copied on the ctx copy stream
 *                       and overlapped with the previous chunk's kernel; the buffer may be
 *                       reused once frb_chunk_done(slot) or frb_sync returns.
 *                       _dev: bytes already resident (16-byte aligned device pointer);
 *                       optional per-read outputs keys_out[r] / rec_off_out[r] (device).
 *   frb_scan_end        file finished: waits, raises queued device errors, exports the file's
 *                       (key,count,first_read) list sorted by first appearance and folds it
 *                       into the running total.
 */
int frb_scan_begin(frb_ctx* ctx, uint32_t file_ordinal, uint64_t read_limit);
int frb_scan_chunk_host(frb_ctx* ctx, const void* host, uint64_t nbytes, uint64_t line_base, int rule);
int frb_scan_chunk_dev(frb_ctx* ctx, const void* dev, uint64_t nbytes, uint64_t line_base, int rule,
                       uint64_t* keys_out_dev, uint64_t* rec_off_out_dev);
int frb_scan_end(frb_ctx* ctx, uint64_t* n_reads, uint64_t* n_unique);
/* Whole .gz file: begin + chunks + end.  Replaces F:159-177.  The deflate stream is inflated ON THE DEVICE (compressed
 * bytes over PCIe, CRC32 + ISIZE of every member verified there); read_limit != 0 (-s), FRB_GZ_DEVICE=0 and streams
 * the device path declines go through zlib on a host thread (pinned double buffers, H2D overlapped with the kernels).
 * A file that ends early, is not gzip or fails its CRC is FRB_ERR_IO on either path. */
int frb_scan_gz(frb_ctx* ctx, const char* path, uint32_t file_ordinal, uint64_t read_limit,
                uint64_t* n_reads, uint64_t* n_unique, uint64_t* raw_bytes);
/* n_files SMALL .gz files (file ordinals ordinals[i]) in one go: laid end to end they are one multi-member gzip
 * stream, inflated by one set of launches; every file is then tallied as itself, with the results frb_scan_gz would
 * give one by one (n_reads / n_unique / raw_bytes: arrays of n_files).  *used_device = 0: declined, nothing changed --
 * call frb_scan_gz per file (which also is how a damaged file gets an error message of its own). */
int frb_scan_gz_batch(frb_ctx* ctx, const char* const* paths, const uint32_t* ordinals, uint32_t n_files,
                      uint64_t* n_reads, uint64_t* n_unique, uint64_t* raw_bytes, int* used_device);
/* A .gz file inflated on the device into host memory (tests, tools).  *used_device = 0: the device path declined
 * the stream (blocks larger than a chunk, '\r' in the text, ...) and nothing was written; frb_scan_gz falls back
 * to zlib on a host thread for such a file.                                                                */
int frb_gz_inflate(frb_ctx* ctx, const char* path, void* host_out, uint64_t cap, uint64_t* nbytes, int* used_device);
/* Span readers: the text of a .gz file inflated ON THE DEVICE and handed out in device memory, for the demux stream
 * (frb_route_push takes the spans).  A context has four slots (0 to 3), one per mate (R1, R2, I1, I2); a slot costs
 * nothing until it is opened.  frb_gz_open closes what the slot held, frb_gz_close frees a slot's thread and buffers
 * (a no-op on a closed slot), frb_destroy closes all of them.
 * frb_gz_read: *dev_text / *n = a span of EXACTLY max_bytes (>= 1) bytes of text, fewer only where the text ends;
 * *eof = 1 when nothing follows the span; *n = 0 after the end.  A span stays valid until the reader has inflated
 * two more pieces (FRB_GZ_PIECE_MB of compressed bytes each), and a copy of it that frb_route_push queued is always
 * done before the reader writes its buffer again.  host_copy: NULL, or max_bytes bytes that receive the span too.
 * *declined = 1: the device path handed the file back -- '\r' in the text, no block start found, not gzip, a
 * truncated file, a CRC-32 / ISIZE mismatch, a read error -- and *n = 0.  *delivered = the text bytes handed out so
 * far (always set); the caller goes on with zlib behind them, and zlib reports any error of the file.  Every read
 * after that says declined again.  Staging overflow is handled inside: the reader starts over with larger staging
 * areas and skips what it handed out.                                                                          */
int frb_gz_open(frb_ctx* ctx, uint32_t slot, const char* path);
int frb_gz_read(frb_ctx* ctx, uint32_t slot, uint64_t max_bytes, const void** dev_text, uint64_t* n, int* eof,
                int* declined, uint64_t* delivered, void* host_copy);
int frb_gz_close(frb_ctx* ctx, uint32_t slot);
/* One buffer -> one gzip member (RFC 1952, zlib's wbits=31 header), encoded ON THE DEVICE (deflate_kernels.cuh:
 * LZ77 + dynamic Huffman per 16 KiB piece, stored where that is not smaller).  host_in: n bytes, pinned or pageable;
 * host_out: cap >= frb_gz_deflate_bound(n) bytes, else FRB_ERR_ARG; *out_n = bytes written.  n = 0 gives the
 * 20-byte empty member.  The same input always gives the same bytes.                                          */
int frb_gz_deflate(frb_ctx* ctx, const void* host_in, uint64_t n, void* host_out, uint64_t cap, uint64_t* out_n);
/* Largest member frb_gz_deflate writes for n bytes: n + 5 per started 16 KiB piece + 20 (no context needed).   */
uint64_t frb_gz_deflate_bound(uint64_t n);
/* One buffer -> one complete BGZF file (the blocked gzip of htslib and bgzip), encoded ON THE DEVICE: blocks of at
 * most 49,152 input bytes, each a gzip member of its own with htslib's 18-byte header (the BC extra field holds the
 * block's size - 1), no back-reference across a block start, then the 28-byte EOF block.  Plain multi-member gzip to
 * any gzip reader.  n = 0 gives the EOF block alone.  cap >= frb_gz_deflate_bgzf_bound(n), else FRB_ERR_ARG.  The
 * same input always gives the same bytes.                                                                      */
int frb_gz_deflate_bgzf(frb_ctx* ctx, const void* host_in, uint64_t n, void* host_out, uint64_t cap, uint64_t* out_n);
/* Largest file frb_gz_deflate_bgzf writes for n bytes: n + 5 per started 16 KiB piece + 28 per started 48 KiB block
 * + 28 (no context needed).                                                                                     */
uint64_t frb_gz_deflate_bgzf_bound(uint64_t n);
/* Per-file results (index = order of frb_scan_end calls) and the merged "total".            */
int frb_file_count(frb_ctx* ctx, uint32_t* n_files);
int frb_file_size(frb_ctx* ctx, uint32_t file_idx, uint64_t* n_unique, uint64_t* n_reads);
int frb_file_export(frb_ctx* ctx, uint32_t file_idx, uint64_t* keys, uint64_t* counts,
                    uint64_t* first_read, uint64_t cap);
int frb_total_finish(frb_ctx* ctx, uint64_t* n_unique); /* sort total by first appearance       */
int frb_total_export(frb_ctx* ctx, uint64_t* keys, uint64_t* counts, uint64_t* first_pos, uint64_t cap);
/* Load a (key,count) list as the total instead of scanning (process() on a caller's dict).  */
int frb_total_load(frb_ctx* ctx, const uint64_t* keys, const uint64_t* counts, uint64_t n);
/* Fold a (key,count,first_pos) list produced elsewhere (another context scanning other files of
 * the same run, F:199-203) into this context's total; first_pos must already be global.
 * A merge into the total table that fails (FRB_ERR_TABLE_FULL) leaves part of the total behind: this call,
 * frb_total_finish and everything built on the total return that error again until frb_reset /
 * frb_resize_tables.                                                                              */
int frb_total_merge(frb_ctx* ctx, const uint64_t* keys, const uint64_t* counts, const uint64_t* first_pos,
                    uint64_t n);
int frb_reset(frb_ctx* ctx); /* forget all files and the total                                 */
/* Key width of the context: 64 (narrow, the default) or 128 (wide, keys of up to 42 symbols).  Implies frb_reset,
 * clears the route table and drops the sample sheet (load it again); frb_reset and frb_resize_tables keep the width.  The *_hi exports return the upper key
 * words in the order of frb_file_export / frb_total_export (all zero on a narrow context); the *2 loads are the
 * narrow calls with upper words added (wide context only).                                                       */
int frb_set_key_width(frb_ctx* ctx, uint32_t bits);
int frb_file_export_hi(frb_ctx* ctx, uint32_t file_idx, uint64_t* keys_hi, uint64_t cap);
int frb_total_export_hi(frb_ctx* ctx, uint64_t* keys_hi, uint64_t cap);
int frb_total_load2(frb_ctx* ctx, const uint64_t* keys, const uint64_t* keys_hi, const uint64_t* counts, uint64_t n);
/* Re-create both unique-key tables with 2^table_log2 slots (implies frb_reset): the host's answer to
 * FRB_ERR_TABLE_FULL -- a Python dict never refuses a key (F:172-177), so the CLI resizes and tallies again. */
int frb_resize_tables(frb_ctx* ctx, uint32_t table_log2);

/* ---- hot path B: mismatch matcher + index-2 orientation ------------------------------------
 * Replaces get_indexes_of_approx_matches F:214-234, analyze_barcode F:237-291,
 * analyze_barcodes_with_rc F:294-351, call_rc_mode_per_id F:354-388 (the sums) and the
 * fan-out process F:391-426.  Runs over the context's total list (frb_total_finish /
 * frb_total_load).  The sheet is given packed: fwd[r] = pack(idx1[r]+"+"+idx2[r]),
 * rc[r] = pack(idx1[r]+"+"+revcomp(idx2[r])) in sheet_mode (case folded, non-ACGTN -> 7);
 * group[r] = dense id of the row's sample NAME (rows sharing a name share a group, F:367).
 * Single-index sheets (l2 = 0) pack idx1 only (extension, parity unpinned).
 *   rc_mode=1: first pass of F:610 -- per key forward and reverse-complement classification
 *     with the cross-ambiguity rule F:336-349, and per-group read sums f_sum/rc_sum.
 *   rc_mode=0: plain pass (F:628); use_rc_rows[r]!=0 selects rc[r] as row r's idx2 (F:618-623).
 * Per-key outputs (host arrays of n_unique entries, any may be NULL): row of the first idx1 /
 * idx2 match or -1, read type, row of the sample or -1.
 */
int frb_sheet_load(frb_ctx* ctx, const uint64_t* fwd, const uint64_t* rc, const int32_t* group,
                   uint32_t n_rows, uint32_t l1, uint32_t l2);
/* Wide context: rows packed as (lo, hi); l1 <= 21, l2 <= 21, l1 + 1 + l2 <= 42.                          */
int frb_sheet_load2(frb_ctx* ctx, const uint64_t* fwd, const uint64_t* fwd_hi, const uint64_t* rc, const uint64_t* rc_hi,
                    const int32_t* group, uint32_t n_rows, uint32_t l1, uint32_t l2);
int frb_match(frb_ctx* ctx, uint32_t n_subs, int rc_mode, const uint8_t* use_rc_rows,
              int32_t* m1_row, int32_t* m2_row, uint8_t* type, int32_t* sample_row,
              int32_t* m2rc_row, uint8_t* type_rc, int32_t* sample_rc_row,
              uint64_t* f_sum, uint64_t* rc_sum);

/* demux_ok of every unique key of the total list and the files that hold a key they should not: the reduction of
 * call_barcodes_correctly_distributed F:504-564 (the regex of F:521-550 is evaluated by the host once per class and
 * file, not per key).  match: (4 + sheet rows) x n_files bytes, row = read type 0/1/3 or 4 + sample row, 0 = the
 * file name does not fit, 1 = fits, 2 = the sample name is not a valid pattern (reported through err_row: the
 * smallest such sample row that really occurs, else INT32_MAX).  file_keys NULL: the per-file lists of this context;
 * else n_files host arrays (file_counts optional: entries with count 0 are skipped).  ok: one byte per unique key in
 * the order of frb_total_export; bad_files: one byte per file.  Uses the classification of the last frb_match. */
int frb_demux_ok(frb_ctx* ctx, const uint8_t* match, uint32_t n_files, const uint64_t* const* file_keys,
                 const uint64_t* const* file_counts, const uint64_t* file_n, uint8_t* ok, uint8_t* bad_files,
                 int32_t* err_row);

/* ---- hot path C: demux record router -------------------------------------------------------
 * Replaces the loop F:774-810 + write_reads F:726-730 (grouping F:719-723).
 *   frb_route_load   results table: packed key -> sink id (from parse_results_file F:645-664
 *                    and the sink selection F:780-801, both done by the host).
 *   frb_route_pair   one record-aligned chunk pair (R1 bytes, R2 bytes; both begin at a record
 *                    start).  Keys come from the R2 headers (F:778).  Whole records of both
 *                    mates are partitioned, stably, into per-sink contiguous regions of
 *                    out_r1 / out_r2 (host, >= the input sizes); sink s of mate m occupies
 *                    [off_m[s], off_m[s+1]) (n_sinks+1 offsets).  Stops at the shorter mate
 *                    (F:777): *n_pairs pairs were routed and consumed_r1/2 bytes of each input
 *                    used; the caller carries the rest into the next call.  final_chunk bit 0 /
 *                    bit 1: the R1 / R2 chunk reaches the end of its file, so a trailing
 *                    partial record of that mate counts as a record (F:719-723).
 */
int frb_route_load(frb_ctx* ctx, const uint64_t* keys, const uint32_t* sink_ids, uint64_t n, uint32_t n_sinks);
/* frb_route_load with the upper words of wide keys (wide context only; the router then parses keys of up to 42
 * symbols from the R2 headers -- from the key mate's headers in a stream of frb_route_set_mates2, index reads
 * included).                                                                                                     */
int frb_route_load2(frb_ctx* ctx, const uint64_t* keys, const uint64_t* keys_hi, const uint32_t* sink_ids, uint64_t n,
                    uint32_t n_sinks);
int frb_route_pair(frb_ctx* ctx, const void* r1, uint64_t r1_bytes, const void* r2, uint64_t r2_bytes,
                   int final_chunk, void* out_r1, void* out_r2, uint64_t* off_r1, uint64_t* off_r2,
                   uint64_t* n_pairs, uint64_t* consumed_r1, uint64_t* consumed_r2, uint64_t* bad_key);
/* The same as a STREAM, two chunk pairs in flight: push queues a chunk pair and returns (H2D, kernels and the D2H
 * of the chunk before run at the same time); the inputs may be cut anywhere -- records that are not complete yet,
 * and the lead of one mate over the other, are carried on the device into the next chunk.  A stream's chunks may
 * not be larger than its first one.  final_chunk bit 0 / 1: the R1 / R2 file ends with this chunk.  Either mate may
 * be host memory (pinned or pageable) or device memory of the context's device, e.g. a span of frb_gz_read (copied
 * device to device on the copy stream); memory of another device is FRB_ERR_ARG.
 *   frb_route_pop  the oldest chunk in flight: *out_r1 / *out_r2 point into pinned memory of the library (valid
 *                   until the chunk after next is pushed), sink s of mate m is out_m[off_m[s], off_m[s + 1]);
 *                   carry_r1 / carry_r2 = bytes pushed so far that are not routed yet.
 *   frb_route_reset a new stream begins (nothing carried).
 *   frb_route_reserve  buffers for chunks of up to chunk_bytes per mate (and a new stream); without it the first
 *                   chunk pushed sets the size.                                                                 */
int frb_route_reset(frb_ctx* ctx);
int frb_route_reserve(frb_ctx* ctx, uint64_t chunk_bytes);
int frb_route_push(frb_ctx* ctx, const void* r1, uint64_t r1_bytes, const void* r2, uint64_t r2_bytes, int final_chunk);
int frb_route_pop(frb_ctx* ctx, void** out_r1, void** out_r2, uint64_t* off_r1, uint64_t* off_r2, uint64_t* n_pairs,
                  uint64_t* carry_r1, uint64_t* carry_r2, uint64_t* bad_key);
/* Gzip mode of the demux stream (on != 0): every chunk is compressed on the device behind the router, and only the
 * compressed bytes cross to the host.  frb_route_pop keeps its meaning, except that out_m[off_m[s], off_m[s + 1]) is
 * one gzip member holding exactly the bytes plain mode returns for sink s of mate m in that chunk; an empty cell stays
 * empty.  Refused with FRB_ERR_STATE while chunks are in flight; kept by frb_route_reset.  frb_route_pair always
 * returns plain bytes.                                                                                          */
int frb_route_set_gzip(frb_ctx* ctx, int on);
/* The output format of the demux stream: FRB_GZ_FORMAT_PLAIN, _GZIP (= frb_route_set_gzip(ctx, 1)) or _BGZF.  In
 * BGZF format out_m[off_m[s], off_m[s + 1]) is a run of whole BGZF blocks (no EOF block) holding exactly the bytes
 * plain mode returns for sink s of mate m in that chunk, so a sink's file is its runs appended chunk after chunk and
 * the EOF block behind them; an empty cell stays empty.  The same rules as frb_route_set_gzip; any other format is
 * FRB_ERR_ARG.                                                                                                  */
int frb_route_set_gz_format(frb_ctx* ctx, int format);
/* Paired (mates = 2, the default) or single-end (mates = 1) demux stream; any other value is FRB_ERR_ARG.  The same
 * rules as frb_route_set_gz_format: refused with FRB_ERR_STATE while chunks are in flight, kept by frb_route_reset.
 * A single-end stream routes the records of R1 alone, each by the key of its own header (the demux rule, F:778
 * applied to the R1 header line); every output format and wide contexts (frb_route_load2) work as in a paired one.
 *   frb_route_push  takes r2 = NULL, r2_bytes = 0 (anything else is FRB_ERR_ARG); only bit 0 of final_chunk counts,
 *                   and a trailing partial record of R1 is routed once it is set.
 *   frb_route_pop   *n_pairs = records routed; *out_r2 = NULL, off_r2 all zero, carry_r2 = 0.
 * frb_route_pair always routes pairs: it saves the setting, routes with mates = 2 and restores it.                */
int frb_route_set_mates(frb_ctx* ctx, int mates);
/* Index reads: a stream of 1 to 4 mates, the keys taken from the headers of mate key_mate (0-based).  The caller
 * orders the mates R1, R2 (absent when single-end), then I1 and / or I2, with key_mate = 1 (R2) or 0 (single-end R1);
 * frb_route_set_mates(ctx, m) is frb_route_set_mates2(ctx, m, m - 1).  Every other mate is parsed for its record
 * offsets alone, and record i of every mate goes to the sink of record i's key; the zip() of F:777 runs over all the
 * mates (a record is routed once every mate has it complete, a trailing partial record counts once its file has
 * ended, and the stream ends once any mate has ended and is used up).  Every output format and wide contexts work as
 * in a paired stream.  mates outside 1..4 or key_mate outside 0..mates-1 is FRB_ERR_ARG; the same rules as
 * frb_route_set_mates otherwise.  The buffers of mates 3 and 4 are allocated when such a stream is first set (or with
 * the stream's other buffers; after frb_route_pair rebuilt the stream for a pair, at the next push).  A stream's
 * histogram keeps one 32-bit counter per sink and mate in the 227 KiB of shared memory a block may have, so a 4-mate stream takes at most 14,528 sinks (3 mates: the usual 16,384): a
 * results table with more is FRB_ERR_ARG, here or at frb_route_load.
 *   frb_route_pushv  in[m] / n[m] = the chunk of mate m (host or device memory, as frb_route_push), for every mate;
 *                    bit m of final_bits: mate m's file ends with this chunk.
 *   frb_route_popv   out[m] = the routed bytes of mate m (pinned memory of the library, valid as for frb_route_pop),
 *                    off[m * (n_sinks + 1) + s] = start of sink s in out[m]; carry[m] (may be NULL) = bytes of mate m
 *                    pushed so far that are not routed yet; *n_records = records routed (of every mate).
 * frb_route_push / frb_route_pop are their one- and two-mate forms; on a stream of 3 or 4 mates they are
 * FRB_ERR_STATE.  frb_route_pair stays two-mate.                                                                   */
int frb_route_set_mates2(frb_ctx* ctx, int mates, int key_mate);
int frb_route_pushv(frb_ctx* ctx, const void* const* in, const uint64_t* n, int final_bits);
int frb_route_popv(frb_ctx* ctx, void** out, uint64_t* off, uint64_t* n_records, uint64_t* carry, uint64_t* bad_key);

/* ---- multi-GPU: merge of the per-rank totals over NCCL (NVLink) ------------------------------
 * One process (or thread) per GPU.  Rank 0 makes the id, the host hands it to every rank.
 * frb_allmerge: all ranks end with the identical merged total (counts add, first_pos min).   */
int frb_nccl_unique_id(char id128[128]);
int frb_nccl_init(frb_ctx* ctx, const char id128[128], int rank, int n_ranks);
int frb_allmerge(frb_ctx* ctx, uint64_t* n_unique);
/* frb_shardmerge: the same merge, but every key ends on ONE rank (its owner by hash): the ranks hold disjoint
 * shares of the merged total, each in first-appearance order; the matcher then runs on the share.           */
int frb_shardmerge(frb_ctx* ctx, uint64_t* n_unique);
/* element-wise sum of a small host array over all ranks (orientation sums of a sharded total, F:354-388) */
int frb_allreduce_u64(frb_ctx* ctx, uint64_t* host_inout, uint64_t n);

/* ---- synthetic input (bench / tests): device twin of frender_b200/synth.py ----------------- */
int frb_synth_load(frb_ctx* ctx, uint64_t seed, uint32_t l1, uint32_t l2, uint32_t n_samples,
                   const uint32_t* emit_i7, const uint32_t* emit_i5, const uint64_t* cdf,
                   uint32_t lane, uint32_t read_len, uint32_t sub_t, uint32_t n_t,
                   uint64_t rand_t, uint64_t hop_t);
int frb_synth_generate(frb_ctx* ctx, uint64_t g0, uint64_t g1, int read_no, void* dev_out,
                       uint64_t cap_bytes, uint64_t* nbytes);

/* ---- measurement --------------------------------------------------------------------------- */
#define FRB_K_SCAN 0   /* parse + pack + count kernel  */
#define FRB_K_EXPORT 1 /* compact + sort + merge       */
#define FRB_K_MATCH 2  /* matcher                      */
#define FRB_K_ROUTE 3  /* demux route + partition      */
#define FRB_K_OTHER 4
#define FRB_K_VERIFY 5 /* line phase of every tile by count (check of the speculative scan) */
#define FRB_K_INFLATE 6 /* device-side gzip inflate */
#define FRB_K_DEFLATE 7 /* device-side gzip writer  */
#define FRB_K_NUM 8
int frb_timer_start(frb_ctx* ctx);            /* CUDA event on the compute stream              */
int frb_timer_stop(frb_ctx* ctx, float* ms);  /* second event, synchronises, elapsed ms        */
int frb_prof_enable(frb_ctx* ctx, int on);    /* per-kernel-class event pairs                  */
int frb_prof_read(frb_ctx* ctx, int kclass, double* ms_total, uint64_t* launches, int reset);
uint64_t frb_launch_count(frb_ctx* ctx);      /* kernels launched by this library on ctx       */

#ifdef __cplusplus
}
#endif
#endif
