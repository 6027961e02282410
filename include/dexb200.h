/* dexb200.h -- C ABI of the B200-native DEXTRACTOR compression hot path (libdexb200.so).
 *
 * Plain C, plain pointers and sizes.  Every entry point names the reference interface it
 * replaces (file:line into the DEXTRACTOR sources).  The reference walks one read at a time
 * through FILE* streams; this library takes whole files (or whole shards of a file) as flat byte
 * buffers and runs hand-written sm_100a CUDA kernels over all entries at once.  The bytes it
 * produces are identical to the reference tools' output.
 *
 * There is NO CPU implementation behind these calls: dx_open fails when no CUDA device is
 * usable, and every compute entry point needs the context it returns.
 *
 * Memory spaces: entry points ending in _dev take DEVICE pointers for bulk data and run on the
 * context's stream without copying; entry points ending in _host take HOST pointers, stage them
 * through pinned memory and include the host<->device copies.  Small results (lengths,
 * statistics, coding tables) always come back in host memory.
 */
#ifndef DEXB200_H
#define DEXB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ----------------------------------------------------------------------------------------------
 *  Status codes.  0 is success; negative values are errors.  The batch tools print
 *  dx_strerror() and exit(1) like the reference's EPRINTF/EXIT convention (DB.h:37-49); an
 *  INTERACTIVE caller copies the text into its Ebuffer and returns the reference's error value.
 * -------------------------------------------------------------------------------------------- */
#define DX_OK          0
#define DX_E_FORMAT   (-1)   /* malformed text: header missing / fields unparsable (QV.c:954-968) */
#define DX_E_CAP      (-2)   /* caller's output buffer too small                                  */
#define DX_E_TRUNC    (-3)   /* compressed input ends early (SYSTEM_READ_ERROR, DB.h:136-139)     */
#define DX_E_KEY      (-4)   /* endian key invalid (undexta.c:156-159, undexar.c:142-145)         */
#define DX_E_LINELEN  (-5)   /* lines of a .quiva entry differ in length (QV.c:792-795)           */
#define DX_E_TOOLONG  (-6)   /* fasta/arrow line longer than MAX_BUFFER-2 (dexta.c:168-172), .quiva entry of >= 2^24 positions */
#define DX_E_ARG      (-7)   /* bad argument                                                      */
#define DX_E_NOMEM    (-8)   /* host or device allocation failed                                  */
#define DX_E_NOGPU    (-9)   /* no usable CUDA device: there is no CPU fallback                   */
#define DX_E_CUDA     (-10)  /* CUDA runtime error (text in dx_strerror)                          */
#define DX_E_CODING   (-11)  /* histogram cannot be coded (fewer than 2 symbols, QV.c:147-220)    */

typedef struct dx_ctx dx_ctx;

/* One context per GPU and per host thread (the reference is single threaded, SURVEY 8b). */
int         dx_open(int device, dx_ctx **ctx);
void        dx_close(dx_ctx *ctx);
const char *dx_strerror(const dx_ctx *ctx);     /* text of the last error on this context       */
int64_t     dx_error_line(const dx_ctx *ctx);   /* 1-based input line of a text error, 0 if n/a */
/* the output size the last call that returned DX_E_CAP needed (0 if it could not tell): allocate that
 * much and call again -- an image has no useful a-priori bound, a single well gap of 2^31 holes is
 * 8.4 MB of 0xff delta bytes (dexta.c:186-193) */
size_t      dx_needed_bytes(const dx_ctx *ctx);
int         dx_sync(dx_ctx *ctx);               /* wait for the context's stream                */
void       *dx_stream(dx_ctx *ctx);             /* the cudaStream_t every _dev call runs on     */

/* Device / pinned-host buffers for C callers that do not link the CUDA runtime themselves. */
void *dx_device_alloc(dx_ctx *ctx, size_t bytes);
void  dx_device_free (dx_ctx *ctx, void *p);
void *dx_pinned_alloc(dx_ctx *ctx, size_t bytes);
void  dx_pinned_free (dx_ctx *ctx, void *p);
int   dx_h2d(dx_ctx *ctx, void *d_dst, const void *h_src, size_t bytes);   /* async on stream */
int   dx_d2h(dx_ctx *ctx, void *h_dst, const void *d_src, size_t bytes);   /* async on stream */
int   dx_d2d(dx_ctx *ctx, void *d_dst, const void *d_src, size_t bytes);   /* async; no overlap */

/* Device memory for sizing windows.  free / total: cudaMemGetInfo of the context's device.  held: the
 * device bytes this context holds now -- its scratch arena, its staging and framing buffers and the live
 * dx_device_alloc blocks.  Any pointer may be NULL. */
int dx_mem_info(dx_ctx *ctx, size_t *free, size_t *total, size_t *held);

/* Where the text of the following calls starts in its file: line0 lines and entry0 entries lie in front
 * of it.  Added to the line and entry numbers of error texts and of dx_error_line, so that a caller that
 * feeds a file window by window reports an error exactly as the whole-file call does.  0, 0 at dx_open. */
int dx_set_origin(dx_ctx *ctx, int64_t line0, int64_t entry0);

/* launches issued by this context since the last reset (for the bench's gpu_launches claim) */
uint64_t dx_launch_count(dx_ctx *ctx, int reset);

/* Test hook: force one of the library's alternative paths on this context (the default for every
 * route is 0 = the product's choice).  Names: "no_fast", "no_spec" (host-planned undex* paths),
 * "exact_index", "exact_pack", "pack2", "two_pass", "chain_scan", "decoder" (1 sequential kernels,
 * 5 warp-per-entry kernel only, 6 lane-per-entry kernel only), "lane_max_rlen", "lane_min_entries",
 * "serial_io" (the *_host calls copy, compute, copy without overlap), "pipe_chunk" (window bytes of
 * the pipelined dx_undexqv_host, so that small files take it too), "no_direct" (dx_undexqv_dev with
 * discovered entries decodes into a scratch image and moves the lines, instead of straight into
 * place), "index_bulk" (the newline index fetches its tiles with cp.async.bulk + mbarrier instead of
 * vector loads: an experiment, value = CTAs per SM), "hist_mode" (how k_qv_hist_run counts a batch: 0 shared atomics, 1 match.any groups, 2 / 3
 * one of each, 4 without the item queue), "arena_cap" (the scratch arena grows to at most this many bytes;
 * beyond, DX_E_NOMEM: how a caller's out-of-memory handling is tested), "debug"; "default" resets all but
 * "debug" and "arena_cap", which dx_open takes from DEXB200_DEBUG and DEXB200_ARENA_CAP.
 * No reference counterpart; nothing in the library reads the environment inside a call. */
int dx_route(dx_ctx *ctx, const char *name, int64_t value);

/* Per-kernel device timing.  While enabled every kernel launch of this context is bracketed by
 * CUDA events on the context's stream; dx_profile_report waits for the stream, writes one line
 * per kernel name -- "name calls total_ms" -- into buf and clears the records. */
int dx_profile(dx_ctx *ctx, int enable);
int dx_profile_report(dx_ctx *ctx, char *buf, size_t cap);

/* ----------------------------------------------------------------------------------------------
 *  2-bit codec: .fasta <-> .dexta and .arrow <-> .dexar
 * -------------------------------------------------------------------------------------------- */
#define DX_FASTA 0      /* Number_Read / Lower_Read / Upper_Read   (DB.c:367-381, 393-416) */
#define DX_ARROW 1      /* Number_Arrow / Letter_Arrow             (DB.c:383-389, 418-441) */

/* Whole-file encode.  Replaces the per-entry loop of dexta.c:100-205 (kind DX_FASTA) and
 * dexar.c:100-211 (DX_ARROW): header parse, line concatenation, well-delta bytes,
 * Number_Read/Number_Arrow + Compress_Read (DB.c:319-338) for every entry, written in file
 * order after the 0x55aa key and the prefix.  out_len <= n/4 + 64 + 17 * entries. */
int dx_dexta_dev (dx_ctx *ctx, int kind, const uint8_t *d_text, size_t n,
                  uint8_t *d_out, size_t cap, size_t *out_len);
int dx_dexta_host(dx_ctx *ctx, int kind, const uint8_t *h_text, size_t n,
                  uint8_t *h_out, size_t cap, size_t *out_len);

/* One part of a file: the entries of d_text[0..n), which starts at an entry header ('>').  lwell_in is
 * the well of the entry in front of the part (0 for the first part), *last_well (if not NULL) returns the
 * well of the part's last entry, for the next part's lwell_in.  with_header = 1 (the first part only):
 * the part also gets the 0x55aa key, plen and prefix, and its first line is checked as dx_dexta_dev
 * checks it.  The parts' outputs concatenated, each part cut in front of a line that starts with '>',
 * are the bytes of dx_dexta_dev on the whole file, which is this call with 0 and 1.  DX_E_CAP and
 * dx_needed_bytes as for dx_dexta_dev. */
int dx_dexta_part_dev(dx_ctx *ctx, int kind, const uint8_t *d_text, size_t n, int32_t lwell_in,
                      int with_header, uint8_t *d_out, size_t cap, size_t *out_len, int32_t *last_well);
/* entries encoded by the last dx_dexta_part_dev / dx_dexta_dev, or decoded by the last
 * dx_undexta_window_dev (the entry0 of the next window's dx_set_origin) */
int64_t dx_last_entries(const dx_ctx *ctx);

/* Whole-file decode.  Replaces undexta.c:130-271 / undexar.c:130-229: endian key (0x55aa,
 * 0xaa55 and, fasta only, the old 0x33cc/0xcc33 16-bit layout), per-entry header text,
 * Uncompress_Read (DB.c:342-363) + Lower_/Upper_Read/Letter_Arrow, `width` symbols per line
 * (-w, default 80), upper = -U. */
int dx_undexta_dev (dx_ctx *ctx, int kind, const uint8_t *d_in, size_t n, int width, int upper,
                    uint8_t *d_out, size_t cap, size_t *out_len);
int dx_undexta_host(dx_ctx *ctx, int kind, const uint8_t *h_in, size_t n, int width, int upper,
                    uint8_t *h_out, size_t cap, size_t *out_len);
/* size of the text dx_undexta_* would produce (header walk only; no payload decode) */
int dx_undexta_size_host(dx_ctx *ctx, int kind, const uint8_t *h_in, size_t n, int width,
                         size_t *out_len);
int dx_undexta_size_dev (dx_ctx *ctx, int kind, const uint8_t *d_in, size_t n, int width,
                         size_t *out_len);

/* One window of a .dexta / .dexar image, for callers that hold only part of the file.  h_head: the image's
 * first min(image size, 6 + plen) bytes on the host (key, plen, prefix).  d_buf (16-byte aligned) holds the
 * image bytes [buf_off, buf_off + buf_n).  The chain starts at image offset cur_in (6 + plen for the first
 * window) with the well well_in (0 for the first); the call decodes every entry from there on that lies
 * wholly in the buffer and stops in front of the first that does not: *cur_out / *well_out are where that
 * entry starts and the well in front of it (the next window's cur_in / well_in).  is_last = 1: the buffer
 * reaches the end of the image, and an entry cut short is DX_E_TRUNC, as for the whole file.
 * DX_E_CAP with *cur_out == cur_in: no entry lies wholly in the buffer (is_last = 0); dx_needed_bytes() is
 * the image offset the buffer has to reach.  DX_E_CAP with *cur_out > cur_in: the text needs
 * dx_needed_bytes() bytes of d_out (d_out may be NULL with cap 0 to ask).  The texts of consecutive windows
 * concatenated are the text of dx_undexta_dev.  Images of the old 0x33cc layout or the other byte order are
 * refused (DX_E_FORMAT): decode them whole. */
int dx_undexta_window_dev(dx_ctx *ctx, int kind, const uint8_t *h_head, size_t head_n, const uint8_t *d_buf,
                          size_t buf_n, int64_t buf_off, int64_t cur_in, int32_t well_in, int is_last,
                          int width, int upper, uint8_t *d_out, size_t cap, size_t *out_len,
                          int64_t *cur_out, int32_t *well_out);

/* Batched in-memory form of the same codec for callers that already hold reads in memory
 * (the Dazzler DB loaders, DB.c:1279-1286, 1414-1432, 1533-1540, 1592-1600 and the dex2DB
 * writer, dex2DB.c:511-566).  Read i is d_src[src_off[i] .. src_off[i]+len[i]) ASCII
 * and goes to d_dst[dst_off[i] .. dst_off[i]+COMPRESSED_LEN(len[i])), or the reverse. */
int dx_compress_reads_dev  (dx_ctx *ctx, int kind, const uint8_t *d_src, const int64_t *d_src_off,
                            const int32_t *d_len, int64_t nreads, uint8_t *d_dst,
                            const int64_t *d_dst_off);
int dx_uncompress_reads_dev(dx_ctx *ctx, int kind, int upper, const uint8_t *d_src,
                            const int64_t *d_src_off, const int32_t *d_len, int64_t nreads,
                            uint8_t *d_dst, const int64_t *d_dst_off);

/* ----------------------------------------------------------------------------------------------
 *  QV coder: .quiva <-> .dexqv
 * -------------------------------------------------------------------------------------------- */

/* The statistics of QVcoding_Scan (QV.c:860-862, 922-1023).  hist index: 0 del, 1 ins, 2 mrg,
 * 3 sub, 4 delRun, 5 subRun.  The run histograms do NOT include the reference's "+1 in every
 * bucket" initialisation (QV.c:934-935); dx_qv_make_coding adds it once, so that histograms of
 * several shards can simply be summed (the multi-GPU allreduce). */
typedef struct
  { uint64_t hist[6][256];
    uint64_t totchar;        /* positions scanned in this shard                                 */
    int64_t  nentries;
    int32_t  delchar;        /* run characters in force at the END of this shard, -1 if none    */
    int32_t  subchar;
    uint64_t sub_prefix[256];/* subHist of the entries up to and including the one at which
                                subchar was fixed (carry for a following shard); else all subs  */
  } dx_qv_stats;

/* What a shard inherits from the shards before it (all zero / -1 for the first shard). */
typedef struct
  { int32_t  delchar, subchar;   /* already fixed by an earlier shard, else -1 */
    uint64_t totchar;            /* positions in earlier shards                */
    uint64_t sub[256];           /* subHist of earlier shards (only read while subchar < 0) */
  } dx_qv_carry;

/* One Huffman table.  Replaces HScheme (QV.c:76-81); the decode LUT lives on the device. */
typedef struct
  { int32_t  type;               /* 0 plain, 2 truncated with escape code 255 */
    uint32_t bits[256];
    int32_t  lens[256];
  } dx_scheme;

/* Replaces QVcoding (QV.h:31-42).  tab: 0 del, 1 dRun, 2 ins, 3 mrg, 4 sub, 5 sRun. */
typedef struct
  { dx_scheme tab[6];
    int32_t   delchar, subchar;  /* -1 if the stream is not run-length coded */
    int32_t   flip;              /* decoder only: file has foreign byte order */
  } dx_qv_coding;

/* Pass 1.  Replaces QVcoding_Scan / QVcoding_Scan1 (QV.c:922-1023 / 866-920) over a whole
 * .quiva text (or one shard of it starting at an entry boundary): frames the entries, checks
 * them the way Read_Lines does (QV.c:751-798), and histograms the five streams.  The framing is
 * kept in the context and reused by dx_qv_encode_dev on the same buffer.  An entry of 2^24 positions
 * or more is refused with DX_E_TOOLONG (the reference takes it; DESIGN section 2). */
int dx_qv_scan_dev(dx_ctx *ctx, const uint8_t *d_text, size_t n, const dx_qv_carry *carry,
                   dx_qv_stats *stats);

/* Replaces Create_QVcoding (QV.c:1029-1169) incl. Huffman/Reheap/Build_Table (QV.c:91-220).
 * Host only, microseconds.  `stats` must be the SUM over all shards (totchar and hist), with
 * delchar/subchar those of the LAST shard. */
int dx_qv_make_coding(const dx_qv_stats *stats, int lossy, dx_qv_coding *coding);

/* Replaces Write_QVcoding (QV.c:1173-1210) / Read_QVcoding (QV.c:1214-1320). */
int dx_qv_write_coding(const dx_qv_coding *coding, const char *prefix, int plen,
                       uint8_t *out, size_t cap, size_t *out_len);
int dx_qv_read_coding (const uint8_t *in, size_t n, dx_qv_coding *coding,
                       char *prefix, int pcap, size_t *used);

/* Pass 2.  Replaces the loop of dexqv.c:114-142 with Compress_Next_QVentry (QV.c:1381-1426):
 * per entry the well-delta bytes, beg/end/qv, then del | tags | ins | mrg | sub.
 * lwell_in is the well of the entry preceding this shard (0 for the first); last_well returns
 * this shard's last well.  h_entry_off, if not NULL, receives nentries+1 byte offsets of the
 * entries inside d_out (an index the decoder can use; it is not part of the file).
 * Memory: the streams are first coded into a scratch image of n + 40 bytes per entry taken from the
 * context's arena, then moved to their offsets (no size pass); a stream that does not fit its room
 * there takes the exact two-pass route.  A coding that assigns a code to the NUL byte is refused
 * (DX_E_CODING): NUL cannot occur inside a line the reference reads with fgets (QV.c:751-798). */
int dx_qv_encode_dev(dx_ctx *ctx, const uint8_t *d_text, size_t n, const dx_qv_coding *coding,
                     int lossy, int32_t lwell_in, uint8_t *d_out, size_t cap, size_t *out_len,
                     int32_t *last_well, int64_t *h_entry_off, int64_t max_entries);

/* The framing kept by dx_qv_scan_dev serves the NEXT dx_qv_encode_dev on the same buffer and is
 * dropped after it (a second encode frames the text again).  The text must not change between the
 * two calls; dx_qv_forget drops the framing explicitly.  dx_qv_last_well: the well number of the last
 * entry of the buffer scanned last -- what the next shard's first well delta is coded against
 * (dexqv.c:128-135); 0 for an empty shard. */
int dx_qv_forget(dx_ctx *ctx);
int dx_qv_last_well(dx_ctx *ctx, int32_t *well);

/* Cutting one .quiva file into shards without parsing it (a line that starts with '@' proves
 * nothing, '@' is QV 31; entries are found by COUNTING lines, QV.c:751-798 reads 6 per entry):
 * *nlines = newlines in d_text[0..n); *skip_off = offset just behind the skip-th newline (0 for
 * skip == 0, -1 when the buffer has fewer).  A rank whose range starts at global line g skips
 * (6 - g % 6) % 6 lines to reach its first entry. */
int dx_text_lines_dev(dx_ctx *ctx, const uint8_t *d_text, size_t n, int64_t skip,
                      int64_t *nlines, int64_t *skip_off);

/* The whole tool on one GPU: scan, make coding, 0x55aa key + coding header, encode.
 * Replaces dexqv.c:59-147.  Like dx_qv_scan_dev, refuses an entry of 2^24 positions or more
 * (DX_E_TOOLONG). */
int dx_dexqv_dev (dx_ctx *ctx, const uint8_t *d_text, size_t n, int lossy,
                  uint8_t *d_out, size_t cap, size_t *out_len);
int dx_dexqv_host(dx_ctx *ctx, const uint8_t *h_text, size_t n, int lossy,
                  uint8_t *h_out, size_t cap, size_t *out_len);

/* Replaces undexqv.c:99-208 with Uncompress_Next_QVentry (QV.c:1428-1481) over the whole file.
 * The file stores no entry lengths, so entry starts are first recovered on the device
 * (candidate headers + verified chain walk); pass h_entry_off/nentries (from dx_qv_encode_dev or
 * a Dazzler .idx, DB.c:2598) to skip that pass.  Offsets are relative to d_in.
 * well_in is the well number of the entry preceding this image (0 for a whole file; for a shard
 * [header][entries of shard r] it is the last well of shard r-1, the decode-side twin of
 * lwell_in above). */
int dx_undexqv_dev (dx_ctx *ctx, const uint8_t *d_in, size_t n, int upper,
                    uint8_t *d_out, size_t cap, size_t *out_len,
                    const int64_t *h_entry_off, int64_t nentries, int32_t well_in);
int dx_undexqv_host(dx_ctx *ctx, const uint8_t *h_in, size_t n, int upper,
                    uint8_t *h_out, size_t cap, size_t *out_len);
/* size of the .quiva text dx_undexqv_* would produce for this file */
int dx_undexqv_size_dev(dx_ctx *ctx, const uint8_t *d_in, size_t n, size_t *out_len);

/* One byte range of a .dexqv image, for callers that cut an image into ranges and decode each on its own
 * GPU (tools/undexqv_mg).  Entry e belongs to the range [a, b) that holds its FIRST byte, its first
 * well-delta byte (undexqv.c:119-208 reads the delta first).  Three calls on one context, in this order,
 * with no other call of the context in between:
 *
 *   dx_undexqv_range_dev       decodes every entry candidate the range needs, speculatively (no chain
 *                              decision yet).  h_head / head_n: the image's first bytes on the host, at
 *                              least its key and coding header (min(image size, 2 + 16384 + 100001)
 *                              bytes are always enough).  d_buf (16-byte aligned) holds the image bytes
 *                              [buf_off, buf_off + buf_n); it must cover [max(a', 4096) - 4096, b) with
 *                              a' = max(a, first) and should hold the tails of the entries that start in
 *                              [a, b).  *first (if not NULL): the byte behind the coding header, where
 *                              the first entry starts.  upper = -U.
 *   dx_undexqv_range_chain     the host walk from the chain position the range before it ended at:
 *                              cur_in / well_in (first / 0 for the range that holds the first entry).
 *                              *cur_out: where the next range's chain starts (>= b; cur_in if no entry
 *                              starts in [cur_in, b)), *well_out: the well of the range's last entry
 *                              (well_in if none).  An entry the candidates miss is read and decoded by
 *                              itself, never an error of a valid image.  DX_E_CAP: an entry's tail lies
 *                              behind the buffer; dx_needed_bytes() is the image offset the buffer has to
 *                              reach -- read that much and start again with dx_undexqv_range_dev.
 *   dx_undexqv_range_text_dev  the text of the range's entries into d_out; DX_E_CAP with
 *                              dx_needed_bytes() = the text's size when cap is smaller (d_out may be
 *                              NULL with cap 0 to ask).  Waits for the context's stream.
 *
 * The text of consecutive ranges, each chained from where the one before it ended, concatenated, is the
 * text of dx_undexqv_dev on the whole image.  Every coding is taken, codes of up to 16 bits included.
 * Images of the old layout or the other byte order are refused (DX_E_FORMAT): decode them whole with
 * dx_undexqv_dev. */
int dx_undexqv_range_dev(dx_ctx *ctx, const uint8_t *h_head, size_t head_n, const uint8_t *d_buf,
                         size_t buf_n, int64_t buf_off, int64_t a, int64_t b, int upper, int64_t *first);
int dx_undexqv_range_chain(dx_ctx *ctx, int64_t cur_in, int32_t well_in, int64_t *cur_out,
                           int32_t *well_out);
int dx_undexqv_range_text_dev(dx_ctx *ctx, uint8_t *d_out, size_t cap, size_t *out_len);

/* Batched Load_QVentry (DB.c:2575-2621, and Load_All... style loaders built on it): the caller knows
 * where every entry's streams start (DAZZ_READ.coff of a Dazzler .qvs, which stores bare streams;
 * or the byte behind beg/end/qv of a .dexqv entry) and how long it is.  Entry i's five lines (del,
 * tag, ins, mrg, sub), each followed by '\n', go to d_out[off[i] ...), off = exclusive prefix sum of
 * 5*(rlen+1), returned in h_out_off[0..nentries] if not NULL; h_end_off[i], if not NULL, receives the
 * first image byte behind entry i (the file position Uncompress_Next_QVentry leaves, QV.c:1428-1481). */
int dx_qv_load_entries_dev(dx_ctx *ctx, const uint8_t *d_in, size_t n, const dx_qv_coding *coding,
                           const int64_t *h_stream_off, const int32_t *h_rlen, int64_t nentries,
                           int upper, uint8_t *d_out, size_t cap, int64_t *h_out_off,
                           int64_t *h_end_off);

/* Where the entries of the last dx_undexqv_dev call were: for callers that keep the reference's
 * per-entry view of a file (the QV.h shim, a Dazzler .idx writer: DAZZ_READ.coff, dex2DB.c:617-621).
 * Off by default; dx_keep_index(ctx,1) makes every following dx_undexqv_dev record one row per
 * entry, dx_last_index copies up to max rows out and returns the number of entries in *count. */
typedef struct
  { int64_t stream_off;      /* first stream byte in the image (just after beg/end/qv)         */
    int64_t end_off;         /* first byte after the entry                                      */
    int64_t text_off;        /* first QV line of the entry in the decoded text                  */
    int32_t rlen, well;
  } dx_index_row;
int dx_keep_index(dx_ctx *ctx, int keep);
int dx_last_index(dx_ctx *ctx, dx_index_row *rows, int64_t max, int64_t *count);

#ifdef __cplusplus
}
#endif
#endif /* DEXB200_H */
