// dx_internal.h -- declarations shared by the host C++ and the CUDA translation units of
// libdexb200.so.  Nothing here is part of the public ABI (that is include/dexb200.h).
#ifndef DX_INTERNAL_H
#define DX_INTERNAL_H

#include <stdint.h>
#include <stddef.h>
#include <cuda_runtime.h>
#include "dexb200.h"

// ---- device-side entry tables (structure of arrays, all in HBM) -----------------------------

// One .quiva entry = header line + 5 equal-length lines (reference QV.c:751-798).
struct QvEntries
{ int64_t  n;            // entries
  int64_t *hdr;          // byte offset of '@'
  int64_t *line0;        // byte offset of the first QV line (delQV); line k at line0 + k*(rlen+1)
  int32_t *rlen;
  int32_t *well, *beg, *end, *qv;
  int32_t *flag;         // 0 ok, 1 header needs the host sscanf path
  int32_t *order;        // ticket -> entry, longest entries first (NULL: file order)
};

// Per-entry encode bookkeeping
struct QvSizes
{ uint32_t *bytes;       // [n][6]: header bytes, del, tags, ins, mrg, sub
  int64_t  *off;         // [n+1] entry byte offsets in the output
};

// Packed code-table entry handed to the encode kernels:
//   bits 0..15 code, 16..20 length, bit 21 "followed by a literal" (escape)
#define DX_ENC_CODE(e)  ((e) & 0xffffu)
#define DX_ENC_LEN(e)   (((e) >> 16) & 0x1fu)
#define DX_ENC_ESC(e)   (((e) >> 21) & 1u)

struct QvEncTables { uint32_t t[6][256]; };          // 6 KB, passed via HBM pointer

// Decode LUTs: 16-bit window -> symbol (reference QV.c:365-372), one 64 KB table per scheme,
// plus the code lengths.  lens[k][255] is the escape length for truncated tables.
struct QvDecTables
{ uint8_t look[6][65536];
  uint8_t lens[6][256];
  int32_t type[6];
};

// Compact two-level decode tables for the parallel decoders (dx_qv_decode5.cu, dx_qv_decode6.cu): the
// top 11 bits of the 16-bit window index prim; codes longer than 11 bits go through a 32-entry
// sub-table.  entry = symbol | length << 8 ; bit 15 of a prim entry = "low 15 bits are a sub-table index".
// One sub-table per distinct 11-bit prefix of a code of 12..16 bits: a scheme has at most 256 codes,
// so 256 sub-tables hold every coding.
#define DX_DEC2_MAXSUB 256
struct QvDecTables2
{ uint16_t prim[6][2048];
  uint16_t sub[6][DX_DEC2_MAXSUB*32];
  int32_t  type[6];
};

// Tables of the parallel decoders (dx_qv_decode5.cu, dx_qv_decode6.cu): 12-bit primary tables that are
// copied to shared memory per stream.  multi: plain streams, up to two symbols per entry (bits 0-4 total
// length incl. the 8 literal bits of an escape, 5-6 symbol count, bit 7 escape, 8-12 length of the
// first code, 16-23 / 24-31 the symbols); single: sym | len << 8.  0 = code longer than 12 bits
// (or no code): look in t2.  abits: predicted stream bits per output position.
struct QvDecTables4
{ uint32_t multi[6][4096];
  uint16_t single[6][4096];
  float    abits[6];
  QvDecTables2 t2;
  // codes longer than 12 bits, sorted by their left-aligned 16-bit value: code16 << 16 | len << 8 | sym
  // (prefix-free codes own disjoint intervals of 16-bit windows, so the code of a window is the last
  // entry at or below it).  Symbols folded onto the escape appear once, as 255.
  uint32_t longs[6][256];
  int32_t  nlong[6];
};

// ---- context --------------------------------------------------------------------------------

struct DxBlock { uint8_t *p; size_t cap, top; };

// Routes: which of the alternative paths a call takes.  All zero = the product's defaults; the
// others exist so that tests can force every path (dx_route, include/dexb200.h).  Read from the
// context, never from the environment, inside the entry points.
enum { DXR_NO_FAST = 0, DXR_NO_SPEC, DXR_EXACT_INDEX, DXR_EXACT_PACK, DXR_PACK2, DXR_TWO_PASS, DXR_CHAIN_SCAN,
       DXR_DECODER,            // 0 default (lane per entry + warp per entry for long ones), 1 sequential,
                               // 5 warp per entry only, 6 lane per entry only
       DXR_LANE_MAX_RLEN,      // > 0: entries longer than this go to the warp-per-entry kernel
       DXR_LANE_MIN_ENTRIES,   // > 0: fewer lane-sized entries than this -> warp per entry for all
       DXR_DEBUG, DXR_SERIAL_IO,
       DXR_PIPE_CHUNK,         // > 0: window size of the pipelined *_host calls in bytes (tests: small files)
       DXR_NO_DIRECT,          // discovered entries: always decode into the scratch image, then assemble
       DXR_INDEX_BULK,         // newline index with cp.async.bulk tiles (experiment); > 1: CTAs per SM
       DXR_HIST_MODE,          // k_qv_hist_run: 0 shared atomics, 1 match.any groups, 2 / 3 one of each, 4 no queue
       DXR_ARENA_CAP,          // > 0: the scratch arena grows to at most this many bytes (DX_E_NOMEM beyond)
       DXR_COUNT };

struct dx_ctx
{ int          device;
  cudaStream_t stream;
  int          sm_count;
  char         err[512];
  int64_t      err_line;
  uint64_t     launches;
  int64_t      route[DXR_COUNT];

  // scratch arena in HBM: a bump allocator over a few cudaMalloc'ed blocks, reset per call and
  // consolidated into one block when a call needed more than one
  DxBlock      blk[32];
  int          nblk;

  // device staging for the *_host entry points (grown on demand, kept)
  uint8_t     *io_in;   size_t io_in_cap;
  uint8_t     *io_out;  size_t io_out_cap;
  // copy streams and events of the pipelined *_host entry points (created on first use)
  size_t       need_bytes;      // output size asked for by the last DX_E_CAP failure (dx_needed_bytes)
  cudaStream_t cs_in, cs_out;
  // host work to do while the next position index runs on the device (called once, before its sync)
  void       (*overlap_fn)(void *);
  void        *overlap_arg;
  cudaEvent_t  pev[40];
  int          npev;

  // per-kernel CUDA-event timing (dx_profile): (name, start, stop) per launch
  int          prof_on;
  void        *prof;           // std::vector<DxProfRec>*

  // pinned host scratch for the small per-call transfers (bump allocated, reset per call)
  uint8_t     *hpin;    size_t hpin_cap, hpin_top, hpin_want;
  void        *hpin_extra;     // one-off blocks handed out when hpin was too small

  // entry index of the last dx_undexqv_dev call, kept on request (dx_keep_index)
  int          keep_index;
  void        *last_index;     // std::vector<dx_index_row>*

  // framing of the last scanned .quiva buffer (reused by the encode pass)
  const uint8_t *qv_text;
  size_t         qv_n;
  QvEntries      qv_ent;
  uint8_t       *qv_store;     // cudaMalloc'ed backing of qv_ent
  size_t         qv_store_cap;

  // the byte range of a .dexqv image between dx_undexqv_range_dev and its _chain / _text_dev calls
  // (QvRange*, dx_api.cpp); live until the next call that resets the arena
  void          *qv_range;
  int            qv_range_live;

  // dx_set_origin: added to the line and entry numbers of error texts and dx_error_line, so that a caller
  // that feeds one file window by window reports what the whole-file call reports
  int64_t        origin_line, origin_entry;
  int64_t        last_entries;  // entries of the last dx_dexta_part_dev / dx_undexta_window_dev
  void          *dev_blocks;    // std::unordered_map<void*, size_t>*: live dx_device_alloc blocks (dx_mem_info)
};

int   dx_fail(dx_ctx *ctx, int code, const char *fmt, ...);
int   dx_cuda_fail(dx_ctx *ctx, cudaError_t e, const char *what);
int   dx_fail_cap(dx_ctx *ctx, size_t need, size_t cap);
void  dx_arena_reset(dx_ctx *ctx);
void *dx_arena_get(dx_ctx *ctx, size_t bytes);        // 256-byte aligned; NULL + error on failure
int   dx_arena_reserve(dx_ctx *ctx, size_t bytes);    // make sure this much is available
void *dx_hpin_get(dx_ctx *ctx, size_t bytes);         // pinned host scratch; NULL + error on failure

#define DX_CUDA(ctx, call) do { cudaError_t e__ = (call); \
    if (e__ != cudaSuccess) return dx_cuda_fail(ctx, e__, #call); } while (0)
void dx_prof_begin(dx_ctx *ctx);
void dx_prof_end(dx_ctx *ctx, const char *what);
#define DX_PROF_BEGIN(ctx) do { if ((ctx)->prof_on) dx_prof_begin(ctx); } while (0)
#define DX_LAUNCHED(ctx, what) do { (ctx)->launches++; cudaError_t e__ = cudaGetLastError(); \
    if ((ctx)->prof_on) dx_prof_end(ctx, what); \
    if (e__ != cudaSuccess) return dx_cuda_fail(ctx, e__, what); } while (0)

// ---- kernels' host launchers (defined in the .cu files) ---------------------------------------

// dx_frame.cu : a few bytes device -> PINNED host memory by a kernel (not by the copy engine), async
int dxk_fetch(dx_ctx *ctx, void *h_pinned, const void *d_src, size_t bytes);

// dx_frame.cu : positions of bytes satisfying a predicate, in order
enum { DX_PRED_NEWLINE = 0, DX_PRED_FASTA_HDR = 1, DX_PRED_QVCAND = 2, DX_PRED_ARCAND = 3 };
int dxk_index_positions(dx_ctx *ctx, int pred, const uint8_t *d_buf, size_t n, size_t first,
                        int64_t **d_pos, int64_t *count);
// order[t] = entry of ticket t, longest first (counting sort on rlen / 512, one CTA)
int dxk_ticket_order(dx_ctx *ctx, const int32_t *d_rlen, int64_t n, int32_t *d_order);
int dxk_qv_entries(dx_ctx *ctx, const uint8_t *d_text, size_t n, const int64_t *d_nl,
                   int64_t nlines, QvEntries ent, int32_t *h_err, uint64_t *h_totchar,
                   int64_t *h_noncanon, int64_t *h_last_nl);

// dx_qv_stats.cu
struct QvProbe                  // device-resident result of the order-dependent prefix rules
{ int32_t  delchar, subchar;
  int64_t  e_del, e_sub;        // first entry whose runs are counted (n if never)
  uint64_t sub_prefix[256];
  uint64_t totchar;
};
int dxk_qv_probe(dx_ctx *ctx, const uint8_t *d_text, QvEntries ent, const dx_qv_carry *carry,
                 QvProbe *h_probe);
int dxk_qv_hist(dx_ctx *ctx, const uint8_t *d_text, QvEntries ent, const QvProbe *h_probe,
                uint64_t *h_hist /*[6][256]*/, int32_t *h_newline_inside);

// dx_qv_encode.cu
int dxk_qv_encode(dx_ctx *ctx, const uint8_t *d_text, size_t text_n, QvEntries ent,
                  const QvEncTables *h_tab,
                  int delchar, int subchar, int lossy, int32_t lwell_in,
                  uint8_t *d_out, size_t cap, size_t *out_len, int32_t *last_well,
                  int64_t *h_entry_off, int64_t max_entries);

// dx_qv_decode.cu
struct QvDecEntry               // host-built table for the decode kernel
{ int64_t out_off;              // where the entry's header text starts in the output
  int64_t text_off;             // where its first QV line starts in the output
  int32_t well, beg, end, qv;
};
// soff: [count][6] = byte offsets of the 5 streams (del, tags, ins, mrg, sub) + entry end
int dxk_qv_walk(dx_ctx *ctx, const uint8_t *d_in, size_t n, const QvDecTables *d_tab,
                int delchar, int subchar, int flip, const int64_t *d_start, const int32_t *d_rlen,
                int64_t count, int64_t *d_soff, int32_t *d_status /*[count]*/);
int dxk_qv_decode(dx_ctx *ctx, const uint8_t *d_in, size_t n, const QvDecTables *d_tab,
                  int delchar, int subchar, int flip, int upper, const QvDecEntry *d_ent,
                  const int64_t *d_soff, int64_t count, const char *d_prefix, int plen,
                  uint8_t *d_out, int32_t *d_status /*[1]*/);

// dx_qv_decode5.cu : one warp per entry, tables resident in shared memory (same contract)
int dxk_qv_decode5(dx_ctx *ctx, const uint8_t *d_in, size_t n, const QvDecTables4 *d_tab,
                   int delchar, int subchar, int upper, int write, int64_t count,
                   const int64_t *d_start, const int32_t *d_rlen, const QvDecEntry *d_ent,
                   const char *d_prefix, int plen, uint8_t *d_out, int64_t *d_soff, int32_t *d_status);

// ... with a per-entry byte limit (an entry that would read past it is reported as bad) and a
// ticket -> entry order (long entries first); either may be NULL.  d_endat (known entry offsets):
// the byte each entry must end at exactly, the next entry's offset -- an entry whose streams end
// anywhere else is reported as bad; NULL: not checked
int dxk_qv_decode5x(dx_ctx *ctx, const uint8_t *d_in, size_t n, const QvDecTables4 *d_tab,
                    int delchar, int subchar, int upper, int write, int64_t count,
                    const int64_t *d_start, const int32_t *d_rlen, const QvDecEntry *d_ent,
                    const char *d_prefix, int plen, uint8_t *d_out, int64_t *d_soff, int32_t *d_status,
                    const int64_t *d_limit, const int32_t *d_order, const int64_t *d_toff,
                    const int64_t *d_endat = NULL);

// dx_qv_decode6.cu : one LANE per entry for tickets [n_coop, count), the warp-per-entry kernel for
// tickets [0, n_coop) (the longest entries); write = 1 or 2
int dxk_qv_decode6x(dx_ctx *ctx, const uint8_t *d_in, size_t n, const QvDecTables4 *d_tab,
                    int delchar, int subchar, int upper, int write, int64_t count,
                    const int64_t *d_start, const int32_t *d_rlen, const QvDecEntry *d_ent,
                    const char *d_prefix, int plen, uint8_t *d_out, int64_t *d_soff, int32_t *d_status,
                    const int64_t *d_limit, const int32_t *d_order, const int64_t *d_toff, int64_t n_coop,
                    const int64_t *d_endat = NULL);

// move speculatively decoded lines (scratch image d_tmp, entry e at d_src[e], < 0 = skip) to their
// final place and write the header lines
int dxk_qv_assemble(dx_ctx *ctx, const uint8_t *d_tmp, size_t tmp_n, const QvDecEntry *d_ent,
                    const int64_t *d_src, int64_t count, const char *d_prefix, int plen, uint8_t *d_out);

// dx_qv_plan.cu : per-entry planning of a .dexqv decode on the device
struct QvPlanArrays              // one row per entry (or candidate), all in HBM
{ int64_t  *fs;                  // first stream byte (after beg/end/qv)
  int32_t  *rlen;                // end - beg; -1 = candidate ruled out
  uint32_t *delta;               // well delta (known-offset path)
  int32_t  *beg, *end, *qv;
};
int dxk_qv_known_prep(dx_ctx *ctx, const uint8_t *d_in, size_t n, const int64_t *d_estart, int64_t count,
                      QvPlanArrays pa, int32_t *d_flag);
int dxk_qv_cand_prep(dx_ctx *ctx, const uint8_t *d_in, size_t n, size_t first, const int64_t *d_q, int64_t count,
                     int span, int minbits, QvPlanArrays pa, uint32_t *d_tlen, int64_t *d_limit,
                     int32_t *d_ffrun, uint8_t *d_last);
int dxk_qv_text_len(dx_ctx *ctx, int64_t count, const int32_t *d_cand, QvPlanArrays pa, const int64_t *d_wpre,
                    const int32_t *d_wells, int32_t well_in, int plen, uint32_t *d_len, int32_t *d_well_out,
                    int32_t *d_flag, const int32_t *d_sel = NULL);
int dxk_qv_direct_prep(dx_ctx *ctx, const int64_t *d_q, int64_t count, QvPlanArrays pa, int32_t *d_rlen_d,
                       uint8_t *d_keep);
int dxk_qv_chain_check(dx_ctx *ctx, const int64_t *d_q, int64_t count, const uint8_t *d_keep, const int32_t *d_rlen_d,
                       const int32_t *d_stat, const int64_t *d_soff, const uint8_t *d_last, const int32_t *d_ffrun,
                       size_t first, size_t n, int32_t *d_flag);
int dxk_qv_build_ent(dx_ctx *ctx, int64_t count, const int32_t *d_cand, QvPlanArrays pa, const int32_t *d_well,
                     const int64_t *d_opre, const uint32_t *d_len, const int64_t *d_toff, QvDecEntry *d_ent,
                     int64_t *d_src, int64_t *d_fs_out, int32_t *d_rlen_out);
// exclusive scan of n 32-bit values into n+1 64-bit prefixes (one CTA)
int dxk_scan_u32(dx_ctx *ctx, const uint32_t *d_in, int64_t n, int64_t *d_prefix);

// dx_pack.cu : .fasta/.arrow <-> 2-bit images
struct FaEntries                // one fasta/arrow entry (structure of arrays in HBM)
{ int64_t  n;
  int64_t *hdr;                 // offset of '>'
  int64_t *seq;                 // offset of the first sequence character
  int64_t *region;              // bytes from seq to the next header / end of text
  int32_t *rlen;                // sequence symbols (newlines excluded)
  int32_t *width;               // length of the first sequence line
  int32_t *well, *beg, *end;
  int32_t *aux;                 // [n][2]: fasta qv,0 ; arrow cnr[0..3] as 4 x uint16
  int32_t *flag;                // bit0 header needs host sscanf, bit1 ragged lines, bit2 line too long
  uint32_t *bytes;              // encoded bytes of the entry (header fields + payload)
  int64_t *off;                 // [n+1] encoded offsets
};
int dxk_fa_measure(dx_ctx *ctx, int kind, const uint8_t *d_text, size_t n, const int64_t *d_hdr,
                   FaEntries ent);
int dxk_fa_offsets(dx_ctx *ctx, int kind, FaEntries ent, int32_t lwell_in, int64_t *h_total);
int dxk_fa_pack(dx_ctx *ctx, int kind, const uint8_t *d_text, size_t n, FaEntries ent,
                int32_t lwell_in, uint8_t *d_out);

// dx_pack2.cu : vectorised forms (used first; the kernels above remain for unusual layouts)
int dxk_fa_measure2(dx_ctx *ctx, int kind, const uint8_t *d_text, size_t n, const int64_t *d_hdr,
                    FaEntries ent, int32_t *d_anyflag);
int dxk_fa_pack2(dx_ctx *ctx, int kind, const uint8_t *d_text, FaEntries ent, int32_t lwell_in, uint8_t *d_out,
                 int32_t *d_err, unsigned long long *d_ticket, int only_leftover);
// dx_pack3.cu : output-centric kernels for entries on the line lattice (width >= 16); entries that
// are not are flagged in *d_leftover and packed by dxk_fa_pack2(only_leftover = 1)
int dxk_fa_pack3(dx_ctx *ctx, int kind, const uint8_t *d_text, size_t n, FaEntries ent, int32_t lwell_in,
                 uint8_t *d_out, int32_t *d_err, int32_t *d_leftover, unsigned long long *d_ticket);

int dxk_compress_reads2(dx_ctx *ctx, int kind, const uint8_t *d_src, const int64_t *d_src_off,
                        const int32_t *d_len, int64_t nreads, uint8_t *d_dst, const int64_t *d_dst_off);
int dxk_uncompress_reads2(dx_ctx *ctx, int kind, int upper, const uint8_t *d_src,
                          const int64_t *d_src_off, const int32_t *d_len, int64_t nreads,
                          uint8_t *d_dst, const int64_t *d_dst_off);

struct PkDecEntry               // table for the unpack kernel
{ int64_t bin_off;              // first payload byte in the image
  int64_t out_off;              // header text start in the output
  int64_t text_off;             // first sequence character in the output
  int32_t well, beg, end;
  int32_t aux[2];               // fasta: qv ; arrow: 4 x uint16 cnr
};
int dxk_pk_walk(dx_ctx *ctx, int fieldbytes, const uint8_t *d_in, size_t n, const int64_t *d_q,
                int64_t count, int64_t *d_end);
int dxk_unpack(dx_ctx *ctx, int kind, int upper, int width, const uint8_t *d_in,
               const PkDecEntry *d_ent, int64_t count, const char *d_prefix, int plen,
               uint8_t *d_out);
int dxk_unpack2(dx_ctx *ctx, int kind, int upper, int width, const uint8_t *d_in, size_t n, const PkDecEntry *d_ent,
                int64_t count, const char *d_prefix, int plen, uint8_t *d_out, unsigned long long *d_ticket);
int dxk_unpack3(dx_ctx *ctx, int kind, int upper, int width, const uint8_t *d_in, size_t n, const PkDecEntry *d_ent,
                int64_t count, const char *d_prefix, int plen, uint8_t *d_out, unsigned long long *d_ticket);
int dxk_pk_cand_prep(dx_ctx *ctx, const uint8_t *d_in, size_t n, size_t first, int fieldbytes, const int64_t *d_q,
                     int64_t count, int64_t *d_end, int32_t *d_ffrun, uint8_t *d_last);
int dxk_pk_layout(dx_ctx *ctx, int kind, const uint8_t *d_in, const int64_t *d_q, const int32_t *d_cand,
                  const int32_t *d_well, int64_t count, int fieldbytes, int plen, int width, uint32_t *d_len,
                  int64_t *d_opre, PkDecEntry *d_ent);
// candidate bookkeeping shared by the .dexta/.dexar/.dexqv chain resolvers: for each candidate
// field position q, the number of 0xff bytes directly before q-1 (capped) and the byte at q-1
struct CandInfo { int32_t ffrun; uint8_t last; uint8_t pad[3]; uint8_t field[16]; };
int dxk_cand_context(dx_ctx *ctx, const uint8_t *d_in, size_t n, size_t first, const int64_t *d_q,
                     int64_t count, int fieldbytes, CandInfo *d_info);
// starts (first well-delta byte of each entry) -> field positions q
int dxk_skip_ff(dx_ctx *ctx, const uint8_t *d_in, size_t n, const int64_t *d_start, int64_t count,
                int64_t *d_q);
// rlen[i] = end - beg read from the 32-bit fields at q[i]
int dxk_field_rlen(dx_ctx *ctx, const uint8_t *d_in, const int64_t *d_q, int64_t count,
                   int32_t *d_rlen);

// batched in-memory reads (DB.c loaders / dex2DB writer)
int dxk_compress_reads(dx_ctx *ctx, int kind, const uint8_t *d_src, const int64_t *d_src_off,
                       const int32_t *d_len, int64_t nreads, uint8_t *d_dst, const int64_t *d_dst_off);
int dxk_uncompress_reads(dx_ctx *ctx, int kind, int upper, const uint8_t *d_src,
                         const int64_t *d_src_off, const int32_t *d_len, int64_t nreads,
                         uint8_t *d_dst, const int64_t *d_dst_off);

#endif
