/* dxcli.h -- shared driver of the six command-line tools (dexta undexta dexar undexar dexqv
 * undexqv).  The tools keep the reference's command lines, flags, file naming and messages
 * (reference dexta.c:25-66, undexta.c:45-93, dexqv.c:24-53, undexqv.c:41-70 and DB.h:79-123), but
 * instead of streaming one read at a time through stdio they hand the WHOLE file to
 * libdexb200.so, which runs it on the GPU -- or, when the file is larger than one window of device
 * memory, one window after the other, with what the format carries from entry to entry (the well, the
 * run characters, the statistics) handed from window to window.  The output is the same bytes either
 * way.  Host code is plain C; there is no CPU codec here. */
#ifndef DXCLI_H
#define DXCLI_H

#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include "dexb200.h"

typedef struct
  { int verbose, keep, pipe, upper, lossy, width; } dx_opts;

struct dx_win;

typedef struct
  { const char *name;        /* program name for messages                       */
    const char *usage;       /* text after "Usage: <name> "                     */
    const char *flags;       /* legal single-letter flags, e.g. "vkiU"          */
    int         has_width;   /* accepts -w<int>                                 */
    const char *src_ext;     /* ".fasta" ...                                    */
    const char *dst_ext;     /* ".dexta" ...                                    */
    const char *help[5];     /* the "      -k: ..." lines of the usage message  */
    /* d_in holds n input bytes on the device; produce *out_len bytes at *d_out (device memory
       obtained with dx_device_alloc, freed by the driver) */
    int (*run)(dx_ctx *ctx, const dx_opts *o, const uint8_t *d_in, size_t n,
               uint8_t **d_out, size_t *out_len);
    /* a file larger than one window: its windows, in file order (see dx_win below); DX_WHOLE asks the
       driver to take the whole file through run after all (an image the windowed calls refuse) */
    int (*stream)(struct dx_win *w);
    double      expand;      /* device bytes a window of input needs, per input byte (default window size) */
  } dx_tool;

#define DX_WHOLE 1

/* A file processed window by window.  The device buffer d holds the input bytes [off, off + n); a
   window is a prefix of it, cut where the format allows.  Bytes behind the cut stay in the buffer for
   the next window (the input is read once, so a pipe works as well as a file).  Host memory is the
   pinned staging buffer, DX_STAGE bytes, whatever the file's size. */
#define DX_STAGE ((size_t) 64 << 20)

typedef struct dx_win
  { dx_ctx        *ctx;
    const dx_opts *o;
    FILE          *in, *out;
    uint8_t       *stage;      /* pinned, DX_STAGE bytes                                         */
    uint8_t       *d;          /* device buffer: input bytes [off, off + n), room for cap        */
    size_t         cap, n;
    int64_t        off;
    int            eof;        /* the input ends at off + n                                      */
    size_t         size;       /* the window size aimed at (halved when a window runs out of memory) */
    uint8_t       *d_out;      /* the windows' output buffer, reused                             */
    size_t         out_cap;
    int64_t        windows;    /* -v: windows run, the largest, the peak of dx_mem_info's held   */
    size_t         largest, peak;
  } dx_win;

void     dx_cli_die(dx_ctx *ctx, int rc);                 /* the tools' error exit */
void     dx_win_fill(dx_win *w, size_t upto);             /* read until the buffer holds upto bytes or the input ends */
void     dx_win_advance(dx_win *w, int64_t to);           /* drop the bytes in front of input offset `to` */
uint8_t *dx_win_out(dx_win *w, size_t need);              /* the output buffer, at least need bytes; NULL: no room */
void     dx_win_write(dx_win *w, const uint8_t *d_src, size_t len);   /* device bytes -> output, in order */
void     dx_win_done(dx_win *w, size_t n);                /* a window of n bytes ran: -v statistics */
void     dx_win_peak(dx_win *w);                          /* sample the device memory held */

/* the windows of the 2-bit tools (dexta / dexar, undexta / undexar) */
int dx_stream_pack(dx_win *w, int kind);
int dx_stream_unpack(dx_win *w, int kind);

int dx_cli_main(const dx_tool *tool, int argc, char *argv[]);

#endif
