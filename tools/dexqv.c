/* dexqv -- .quiva -> .dexqv (per-file Huffman + run-length coding of the five QV streams).
 * Same command line, flags and file format as the reference's dexqv (dexqv.c:22-53); the work is
 * done by libdexb200.so on the GPU (see dxcli.h). */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "dxcli.h"

static int run(dx_ctx *ctx, const dx_opts *o, const uint8_t *d_in, size_t n,
               uint8_t **d_out, size_t *out_len)
{ size_t cap = 3*n + 200000;            /* worst case: every symbol escaped (24 bits) */
  *d_out = (uint8_t *) dx_device_alloc(ctx,cap);
  if (*d_out == NULL) return DX_E_NOMEM;
  return dx_dexqv_dev(ctx,d_in,n,o->lossy,*d_out,cap,out_len);
}

/* Two passes over the windows, as the reference makes two over the file (QVcoding_Scan, then rewind):
   1. windows cut behind a multiple of 6 lines (QV.c:751-798 reads 6 per entry; '@' is QV 31, so a
      line is never recognised by its first byte), each scanned with what the windows before it carry
      (the run characters, the positions, the sub histogram), the histograms summed;
   2. the coding header once, then the same windows again, each encoded against the last well of the
      window before it. */
static int stream(dx_win *w)
{ dx_ctx *ctx = w->ctx;
  dx_qv_stats  *st  = (dx_qv_stats *) calloc(1,sizeof(dx_qv_stats));
  dx_qv_stats  *tot = (dx_qv_stats *) calloc(1,sizeof(dx_qv_stats));
  dx_qv_carry  *cy  = (dx_qv_carry *) calloc(1,sizeof(dx_qv_carry));
  dx_qv_coding *cd  = (dx_qv_coding *) calloc(1,sizeof(dx_qv_coding));
  uint8_t *head = (uint8_t *) malloc(100000), *hdr = (uint8_t *) malloc(2 + 16384 + 100000);
  size_t head_n = 0, hlen = 0, ncut = 0, maxcut = 1024;
  int64_t *cut = (int64_t *) malloc(maxcut*sizeof(int64_t)), line0 = 0;
  int rc;
  if (!st || !tot || !cy || !cd || !head || !hdr || !cut) dx_cli_die(ctx,DX_E_NOMEM);
  cy->delchar = cy->subchar = -1;

  /* ---- 1. statistics ---------------------------------------------------------------------------- */
  for (;;)
    { size_t lim = w->size, n;
      dx_win_fill(w,lim);
      if (w->n == 0) break;
      if (w->off == 0)
        { head_n = (w->n < 100000) ? w->n : 100000;
          if ((rc = dx_d2h(ctx,head,w->d,head_n)) != DX_OK || (rc = dx_sync(ctx)) != DX_OK) dx_cli_die(ctx,rc);
        }
      for (;;)
        { int64_t lines = 0, at = -1;
          n = (w->n < lim) ? w->n : lim;
          if (w->eof && n == w->n) break;                  /* the rest of the file */
          if ((rc = dx_text_lines_dev(ctx,w->d,n,0,&lines,NULL)) != DX_OK) dx_cli_die(ctx,rc);
          if (lines >= 6)
            { if ((rc = dx_text_lines_dev(ctx,w->d,n,6*(lines/6),&lines,&at)) != DX_OK) dx_cli_die(ctx,rc);
              n = (size_t) at;
              break;
            }
          lim *= 2;                                        /* an entry longer than the window */
          dx_win_fill(w,lim);
        }
      if ((rc = dx_set_origin(ctx,line0,line0/6)) != DX_OK) dx_cli_die(ctx,rc);
      rc = dx_qv_scan_dev(ctx,w->d,n,cy,st);
      if (rc == DX_E_NOMEM && w->size > ((size_t) 64 << 10)) { w->size /= 2; continue; }
      if (rc != DX_OK) dx_cli_die(ctx,rc);
      for (int k = 0; k < 6; k++)
        for (int x = 0; x < 256; x++) tot->hist[k][x] += st->hist[k][x];
      tot->totchar += st->totchar; tot->nentries += st->nentries;
      cy->delchar = st->delchar; cy->subchar = st->subchar; cy->totchar += st->totchar;
      memcpy(cy->sub,st->sub_prefix,sizeof(cy->sub));
      line0 += 6*st->nentries;
      if (ncut == maxcut && (cut = (int64_t *) realloc(cut,(maxcut *= 2)*sizeof(int64_t))) == NULL)
        dx_cli_die(ctx,DX_E_NOMEM);
      cut[ncut++] = w->off + (int64_t) n;
      dx_win_done(w,n);
      dx_win_advance(w,w->off + (int64_t) n);
    }
  if ((rc = dx_set_origin(ctx,0,0)) != DX_OK) dx_cli_die(ctx,rc);

  /* ---- the coding and its header (dexqv.c:59-112) --------------------------------------------------- */
  tot->delchar = cy->delchar; tot->subchar = cy->subchar;
  if (tot->nentries == 0)
    { fprintf(stderr,"dexqv: no entries in .quiva input\n"); exit (1); }
  if (dx_qv_make_coding(tot,w->o->lossy,cd) != DX_OK)
    { fprintf(stderr,"dexqv: a QV stream has fewer than two distinct symbols: cannot build a code\n"); exit (1); }
  { const uint8_t *sl = (const uint8_t *) memchr(head + 1,'/',head_n - 1);
    const uint16_t key = 0x55aa;
    if (sl == NULL) { fprintf(stderr,"dexqv: Header line incorrectly formatted ?\n"); exit (1); }
    memcpy(hdr,&key,2);
    if (dx_qv_write_coding(cd,(const char *) head,(int) (sl - head),hdr + 2,2 + 16384 + 100000 - 2,&hlen) != DX_OK)
      { fprintf(stderr,"dexqv: could not write the coding header\n"); exit (1); }
    hlen += 2;
    if (fwrite(hdr,1,hlen,w->out) != hlen) { fprintf(stderr,"dexqv: System error, write failed!\n"); exit (2); }
  }
  /* the buffer is refilled with other text at the same address: the last scan's framing must go */
  if ((rc = dx_qv_forget(ctx)) != DX_OK) dx_cli_die(ctx,rc);

  /* ---- 2. encode, window by window ------------------------------------------------------------------ */
  if (fseeko(w->in,0,SEEK_SET) != 0) { fprintf(stderr,"dexqv: System error, read failed!\n"); exit (2); }
  w->off = 0; w->n = 0; w->eof = 0;
  int32_t lwell = 0;
  for (size_t k = 0; k < ncut; )
    { size_t n = (size_t) (cut[k] - w->off), m = 0;
      int32_t last = 0;
      dx_win_fill(w,n);
      if (w->n < n) dx_cli_die(ctx,DX_E_TRUNC);           /* the file changed under us */
      for (;;)
        { uint8_t *d_out = dx_win_out(w,n/2 + ((size_t) 1 << 20));
          rc = d_out ? dx_qv_encode_dev(ctx,w->d,n,cd,w->o->lossy,lwell,d_out,w->out_cap,&m,&last,NULL,0) : DX_E_NOMEM;
          if (rc == DX_E_CAP)                              /* worst case: every symbol escaped (24 bits) */
            { d_out = dx_win_out(w,3*n + 200000);
              rc = d_out ? dx_qv_encode_dev(ctx,w->d,n,cd,w->o->lossy,lwell,d_out,w->out_cap,&m,&last,NULL,0) : DX_E_NOMEM;
            }
          if (rc != DX_E_NOMEM || n <= ((size_t) 64 << 10)) break;
          /* the encode needs more than the scan did: the front half of the window, cut behind a multiple
             of 6 lines (the bytes do not depend on where the windows end) */
          int64_t lines = 0, at = -1;
          if ((rc = dx_text_lines_dev(ctx,w->d,n/2,0,&lines,NULL)) != DX_OK) dx_cli_die(ctx,rc);
          if (lines < 6) { rc = DX_E_NOMEM; break; }
          if ((rc = dx_text_lines_dev(ctx,w->d,n/2,6*(lines/6),&lines,&at)) != DX_OK) dx_cli_die(ctx,rc);
          n = (size_t) at;
        }
      if (rc != DX_OK) dx_cli_die(ctx,rc);
      dx_win_peak(w);
      dx_win_write(w,w->d_out,m);
      lwell = last;
      dx_win_advance(w,w->off + (int64_t) n);
      if (w->off == cut[k]) k++;
    }
  free(st); free(tot); free(cy); free(cd); free(head); free(hdr); free(cut);
  return DX_OK;
}

int main(int argc, char *argv[])
{ static const dx_tool tool =
    { "dexqv", "[-vkl] <path:quiva> ...", "vkl", 0, ".quiva", ".dexqv",
      { "      -k: do *not* remove the .quiva file on completion.",
        "      -l: use lossy compression (not recommended).", NULL, NULL, NULL }, run, stream, 8.0 };
  return dx_cli_main(&tool,argc,argv);
}
