/* undexqv -- .dexqv -> .quiva.
 * Same command line, flags and file format as the reference's undexqv (undexqv.c:18-70); the
 * work is done by libdexb200.so on the GPU (see dxcli.h). */
#include <stdint.h>
#include "dxcli.h"

#define BACK     4096                          /* what a range decode looks back at, in front of the range */
#define HEADMAX  ((size_t) 2 + 16384 + 100001) /* key + coding header + prefix, at most */

static int run(dx_ctx *ctx, const dx_opts *o, const uint8_t *d_in, size_t n,
               uint8_t **d_out, size_t *out_len)
{ size_t cap = 0;
  int rc = dx_undexqv_size_dev(ctx,d_in,n,&cap);
  if (rc != DX_OK) return rc;
  *d_out = (uint8_t *) dx_device_alloc(ctx,cap + 64);
  if (*d_out == NULL) return DX_E_NOMEM;
  return dx_undexqv_dev(ctx,d_in,n,o->upper,*d_out,cap + 64,out_len,NULL,0,0);
}

/* Byte ranges of one image on one context (dx_undexqv_range_*): a window decodes the entries that start
   in [cur, b), b a quarter of the buffer in front of its end, so that their tails are in it; the chain
   position and well it ends at start the next window, whose buffer begins BACK bytes in front of it. */
static int stream(dx_win *w)
{ dx_ctx *ctx = w->ctx;
  static uint8_t head[HEADMAX];
  size_t head_n;
  int rc;
  dx_win_fill(w,w->size);
  head_n = (w->n < HEADMAX) ? w->n : HEADMAX;
  if ((rc = dx_d2h(ctx,head,w->d,head_n)) != DX_OK || (rc = dx_sync(ctx)) != DX_OK) dx_cli_die(ctx,rc);
  if (head_n < 2 || head[0] != 0xaa || head[1] != 0x55)
    return DX_WHOLE;                           /* old layout or other byte order */
  int64_t cur = -1, first = 0;
  int32_t well = 0;
  for (;;)
    { size_t lim = w->size, m = 0, buf_n;
      int64_t cur_out = 0;
      int32_t well_out = 0;
      int last, finished = 0;
      dx_win_fill(w,lim);
      for (;;)
        { buf_n = (w->n < lim) ? w->n : lim;
          last = w->eof && buf_n == w->n;
          const int64_t a = (cur < 0) ? 0 : cur, b = last ? w->off + (int64_t) buf_n : w->off + (int64_t) (buf_n - buf_n/4);
          if (last && a >= b) { finished = 1; break; }   /* the window before ended at the image's end */
          if (b <= a) { lim *= 2; dx_win_fill(w,lim); continue; }
          rc = dx_undexqv_range_dev(ctx,head,head_n,w->d,buf_n,w->off,a,b,w->o->upper,&first);
          if (rc == DX_OK) rc = dx_sync(ctx);
          if (rc == DX_E_NOMEM && w->size > ((size_t) 64 << 10)) { w->size /= 2; lim = w->size; continue; }
          if (rc != DX_OK) dx_cli_die(ctx,rc);
          rc = dx_undexqv_range_chain(ctx,cur < 0 ? first : cur,well,&cur_out,&well_out);
          if (rc == DX_E_CAP)                  /* an entry's tail lies behind the buffer */
            { const size_t need = dx_needed_bytes(ctx) - (size_t) w->off;
              if (last) dx_cli_die(ctx,DX_E_TRUNC);
              lim = (need > 2*lim) ? need : 2*lim;
              dx_win_fill(w,lim);
              continue;
            }
          if (rc != DX_OK) dx_cli_die(ctx,rc);
          if (last && cur_out != w->off + (int64_t) buf_n) dx_cli_die(ctx,DX_E_TRUNC);
          rc = dx_undexqv_range_text_dev(ctx,NULL,0,&m);
          if (rc == DX_E_CAP)
            { uint8_t *d_out = dx_win_out(w,dx_needed_bytes(ctx) + 64);
              rc = d_out ? dx_undexqv_range_text_dev(ctx,d_out,w->out_cap,&m) : DX_E_NOMEM;
            }
          if (rc == DX_E_NOMEM && w->size > ((size_t) 64 << 10)) { w->size /= 2; lim = w->size; continue; }
          if (rc != DX_OK) dx_cli_die(ctx,rc);
          break;
        }
      if (finished) break;
      dx_win_done(w,buf_n);
      dx_win_write(w,w->d_out,m);
      if (last) break;
      cur = cur_out; well = well_out;
      dx_win_advance(w,((cur > BACK) ? cur - BACK : 0) & ~(int64_t) 15);
    }
  return DX_OK;
}

int main(int argc, char *argv[])
{ static const dx_tool tool =
    { "undexqv", "[-vkU] <path:dexqv> ...", "vkU", 0, ".dexqv", ".quiva",
      { "      -k: do *not* remove the .dexqv file on completion.",
        "      -U: use uppercase letters (default is lower case).", NULL, NULL, NULL }, run, stream, 12.0 };
  return dx_cli_main(&tool,argc,argv);
}
