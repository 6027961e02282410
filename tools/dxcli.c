/* dxcli.c -- see dxcli.h */
#define _GNU_SOURCE
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <strings.h>
#include <sys/stat.h>
#include <unistd.h>
#include "dxcli.h"

static const char *Prog;

static void die(dx_ctx *ctx, int rc)
{ if (rc == DX_E_TRUNC)                       /* SYSTEM_READ_ERROR, DB.h:136-139 */
    { fprintf(stderr,"%s: System error, read failed!\n",Prog);
      exit (2);
    }
  fprintf(stderr,"%s: %s\n",Prog,ctx ? dx_strerror(ctx) : "cannot open a CUDA device (no CPU fallback)");
  exit (1);
}

void dx_cli_die(dx_ctx *ctx, int rc) { die(ctx,rc); }

#define DXC(call) do { int rc__ = (call); if (rc__ != DX_OK) die(w->ctx,rc__); } while (0)

/* ---- windows --------------------------------------------------------------------------------- */

#define MINWIN ((size_t) 64 << 10)             /* a window below this is only overhead */

static void write_failed(void)
{ fprintf(stderr,"%s: System error, write failed!\n",Prog); exit (2); }

/* room for cap input bytes; 0 when the device has none */
static int grow(dx_win *w, size_t cap)
{ uint8_t *d = (uint8_t *) dx_device_alloc(w->ctx,cap + 64);
  if (d == NULL) return 0;
  if (w->n > 0) DXC(dx_d2d(w->ctx,d,w->d,w->n));
  DXC(dx_sync(w->ctx));
  dx_device_free(w->ctx,w->d);
  w->d = d; w->cap = cap;
  return 1;
}

void dx_win_fill(dx_win *w, size_t upto)
{ while (!w->eof && w->n < upto)
    { if (w->n == w->cap)                      /* room doubles up to what is asked for */
        { size_t c = 2*w->cap > DX_STAGE ? 2*w->cap : DX_STAGE;
          if (!grow(w,c < upto ? c : upto)) die(w->ctx,DX_E_NOMEM);   /* one entry does not fit */
        }
      size_t want = upto - w->n;
      if (want > w->cap - w->n) want = w->cap - w->n;
      if (want > DX_STAGE) want = DX_STAGE;
      size_t got = fread(w->stage,1,want,w->in);
      if (got > 0)
        { DXC(dx_h2d(w->ctx,w->d + w->n,w->stage,got));
          DXC(dx_sync(w->ctx));
          w->n += got;
        }
      if (got < want)
        { if (ferror(w->in)) { fprintf(stderr,"%s: System error, read failed!\n",Prog); exit (2); }
          w->eof = 1;
        }
    }
}

void dx_win_advance(dx_win *w, int64_t to)
{ if (to <= w->off) return;
  size_t k = (size_t) (to - w->off), tail = w->n - k;
  for (size_t at = 0; at < tail; at += k)      /* copies of at most k bytes never overlap */
    DXC(dx_d2d(w->ctx,w->d + at,w->d + k + at,(tail - at < k) ? tail - at : k));
  DXC(dx_sync(w->ctx));
  w->n = tail; w->off = to;
}

uint8_t *dx_win_out(dx_win *w, size_t need)
{ if (need > w->out_cap)
    { dx_device_free(w->ctx,w->d_out);
      w->out_cap = 0;
      if ((w->d_out = (uint8_t *) dx_device_alloc(w->ctx,need)) == NULL) return NULL;
      w->out_cap = need;
    }
  return w->d_out;
}

void dx_win_write(dx_win *w, const uint8_t *d_src, size_t len)
{ for (size_t at = 0; at < len; at += DX_STAGE)
    { size_t part = (len - at < DX_STAGE) ? len - at : DX_STAGE;
      DXC(dx_d2h(w->ctx,w->stage,d_src + at,part));
      DXC(dx_sync(w->ctx));
      if (fwrite(w->stage,1,part,w->out) != part) write_failed();
    }
}

void dx_win_peak(dx_win *w)
{ size_t held = 0;
  DXC(dx_mem_info(w->ctx,NULL,NULL,&held));
  if (held > w->peak) w->peak = held;
}

void dx_win_done(dx_win *w, size_t n)
{ w->windows += 1;
  if (n > w->largest) w->largest = n;
  dx_win_peak(w);
}

/* input offset of the last '>' that starts a line in the first lim bytes of the buffer (0 if none) */
static int64_t last_header(dx_win *w, size_t lim)
{ const size_t chunk = (size_t) 1 << 20;
  size_t hi = lim;
  while (hi > 1)
    { size_t lo = (hi > chunk) ? hi - chunk : 0;
      DXC(dx_d2h(w->ctx,w->stage,w->d + lo,hi - lo));
      DXC(dx_sync(w->ctx));
      size_t len = hi - lo;
      const uint8_t *p;
      while (len > 1 && (p = (const uint8_t *) memrchr(w->stage + 1,'>',len - 1)) != NULL)
        { if (p[-1] == '\n') return w->off + (int64_t) (lo + (size_t) (p - w->stage));
          len = (size_t) (p - w->stage);
        }
      if (lo == 0) break;
      hi = lo + 1;                             /* the byte at lo is looked at with the one in front of it */
    }
  return 0;
}

/* .fasta / .arrow: a line that starts with '>' is always a header, so a window ends in front of the
   last one it holds, and the next part starts there with the well of the part before it */
int dx_stream_pack(dx_win *w, int kind)
{ dx_ctx *ctx = w->ctx;
  int32_t lwell = 0;
  int64_t entries = 0;
  int first = 1;
  for (;;)
    { size_t lim = w->size;
      int64_t cut;
      dx_win_fill(w,lim);
      if (w->n == 0) break;
      for (;;)
        { if (w->eof && w->n <= lim) { cut = w->off + (int64_t) w->n; break; }
          if ((cut = last_header(w,w->n < lim ? w->n : lim)) > w->off) break;
          lim *= 2;                            /* an entry longer than the window */
          dx_win_fill(w,lim);
        }
      const size_t n = (size_t) (cut - w->off);
      size_t cap = n/3 + 200000, m = 0;
      int32_t last = 0;
      int rc;
      DXC(dx_set_origin(ctx,0,entries));
      for (;;)
        { uint8_t *d_out = dx_win_out(w,cap);
          rc = d_out ? dx_dexta_part_dev(ctx,kind,w->d,n,lwell,first,d_out,w->out_cap,&m,&last) : DX_E_NOMEM;
          if (rc != DX_E_CAP || dx_needed_bytes(ctx) <= w->out_cap) break;
          cap = dx_needed_bytes(ctx) + 64;
        }
      if (rc == DX_E_NOMEM && w->size > MINWIN && n > MINWIN)
        { w->size /= 2; continue; }            /* the same window again, smaller */
      if (rc != DX_OK) die(ctx,rc);
      entries += dx_last_entries(ctx);
      dx_win_done(w,n);
      dx_win_write(w,w->d_out,m);
      lwell = last; first = 0;
      dx_win_advance(w,cut);
    }
  return dx_set_origin(ctx,0,0);
}

/* .dexta / .dexar: the chain of entries from the position and well the window before it ended at */
int dx_stream_unpack(dx_win *w, int kind)
{ dx_ctx *ctx = w->ctx;
  uint8_t head[6 + 100001];
  size_t head_n;
  int32_t plen = 0;
  dx_win_fill(w,w->size);
  head_n = (w->n < sizeof(head)) ? w->n : sizeof(head);
  DXC(dx_d2h(ctx,head,w->d,head_n));
  DXC(dx_sync(ctx));
  if (head_n >= 6) memcpy(&plen,head + 2,4);
  if (head_n < 6 || head[0] != 0xaa || head[1] != 0x55 || plen < 0 || (size_t) plen + 6 > head_n)
    return DX_WHOLE;                           /* old layout, other byte order, no key: as a whole */
  int64_t cur = 6 + plen;
  int32_t well = 0;
  dx_win_out(w,5*w->size + ((size_t) 1 << 20));   /* the text of a window is about four times its image */
  for (;;)
    { size_t lim = w->size, m = 0;
      int64_t cur_out = cur;
      int32_t well_out = well;
      int rc;
      dx_win_fill(w,lim);
      for (;;)
        { const size_t buf_n = (w->n < lim) ? w->n : lim;
          const int last = w->eof && buf_n == w->n;
          rc = dx_undexta_window_dev(ctx,kind,head,(size_t) plen + 6,w->d,buf_n,w->off,cur,well,last,w->o->width,
                                     w->o->upper,w->d_out,w->out_cap,&m,&cur_out,&well_out);
          if (rc == DX_E_CAP && cur_out == cur)          /* no whole entry in the window: read on */
            { const size_t need = dx_needed_bytes(ctx) - (size_t) w->off;
              lim = (need > 2*lim) ? need : 2*lim;
              dx_win_fill(w,lim);
              continue;
            }
          if (rc == DX_E_CAP)                            /* the text needs a larger output buffer */
            { if (dx_win_out(w,dx_needed_bytes(ctx) + 64) != NULL) continue;
              rc = DX_E_NOMEM;
            }
          if (rc == DX_E_NOMEM && lim > MINWIN && buf_n > MINWIN)
            { w->size /= 2; lim = w->size; continue; }
          if (rc != DX_OK) die(ctx,rc);
          dx_win_done(w,buf_n);
          break;
        }
      dx_win_write(w,w->d_out,m);
      const int done = w->eof && cur_out == w->off + (int64_t) w->n;
      cur = cur_out; well = well_out;
      dx_win_advance(w,cur);
      if (done) break;
    }
  return DX_OK;
}

/* whole stream into pinned host memory */
static uint8_t *slurp(dx_ctx *ctx, FILE *f, size_t *n)
{ size_t cap = (size_t) 1 << 26, len = 0;
  uint8_t *buf = (uint8_t *) dx_pinned_alloc(ctx,cap);
  if (buf == NULL) die(ctx,DX_E_NOMEM);
  if (f != stdin && fseeko(f,0,SEEK_END) == 0)
    { off_t sz = ftello(f);
      rewind(f);
      if (sz > 0 && (size_t) sz + 64 > cap)
        { dx_pinned_free(ctx,buf);
          cap = (size_t) sz + 64;
          buf = (uint8_t *) dx_pinned_alloc(ctx,cap);
          if (buf == NULL) die(ctx,DX_E_NOMEM);
        }
    }
  while (1)
    { size_t got = fread(buf+len,1,cap-len,f);
      len += got;
      if (got == 0) break;
      if (len == cap)
        { uint8_t *nb = (uint8_t *) dx_pinned_alloc(ctx,2*cap);
          if (nb == NULL) die(ctx,DX_E_NOMEM);
          memcpy(nb,buf,len);
          dx_pinned_free(ctx,buf);
          buf = nb; cap *= 2;
        }
    }
  *n = len;
  return buf;
}

/* <dir>/<root><ext> from a command-line name, the way PathTo/Root/Catenate do (DB.c:112-181):
   the extension is stripped only if present (compared without case) */
static char *file_name(const char *arg, const char *strip, const char *ext)
{ size_t la = strlen(arg), ls = strlen(strip);
  char *out = (char *) malloc(la + strlen(ext) + 16);
  const char *base = strrchr(arg,'/');
  size_t pre = 0;
  if (base == NULL)                      /* PathTo gives "." for a bare name: "./<root><ext>" */
    { strcpy(out,"./"); pre = 2; base = arg; }
  else
    base = base+1;
  strcpy(out+pre,arg);
  if (strlen(base) > ls && strcasecmp(arg+la-ls,strip) == 0)
    out[pre+la-ls] = '\0';
  strcat(out,ext);
  return out;
}

static char *root_name(const char *arg, const char *strip)
{ char *f = file_name(arg,strip,"");
  char *b = strrchr(f,'/');
  char *r = strdup(b == NULL ? f : b+1);
  free(f);
  return r;
}

/* the whole input on the device through tool->run, as one window */
static void run_whole(const dx_tool *tool, const dx_opts *o, dx_win *w)
{ uint8_t *d_out = NULL;
  size_t m = 0;
  int rc;
  dx_win_fill(w,(size_t) -1);
  if ((rc = tool->run(w->ctx,o,w->d,w->n,&d_out,&m)) != DX_OK) die(w->ctx,rc);
  dx_win_done(w,w->n);
  dx_win_write(w,d_out,m);
  dx_device_free(w->ctx,d_out);
}

/* windows of the input, in file order, until its end */
static void run_windows(const dx_tool *tool, const dx_opts *o, dx_ctx *ctx, FILE *in, FILE *out, size_t window,
                        off_t fsize)
{ dx_win w;
  memset(&w,0,sizeof(w));
  w.ctx = ctx; w.o = o; w.in = in; w.out = out; w.size = window;
  if ((w.stage = (uint8_t *) dx_pinned_alloc(ctx,DX_STAGE)) == NULL) die(ctx,DX_E_NOMEM);
  if (fsize > 0)                               /* no room for the window: a smaller one */
    while (!grow(&w,(size_t) fsize < w.size ? (size_t) fsize : w.size))
      { if (w.size <= MINWIN) die(ctx,DX_E_NOMEM);
        w.size /= 2;
      }
  if (fsize < 0)                               /* a pipe: one window if it ends within one */
    { dx_win_fill(&w,window);
      if (w.eof) { run_whole(tool,o,&w); goto done; }
    }
  if (tool->stream(&w) == DX_WHOLE)
    run_whole(tool,o,&w);
done:
  if (o->verbose && w.windows > 1)
    { fprintf(stderr,"  %lld windows, largest %zu bytes, peak device memory held %zu bytes\n",
              (long long) w.windows,w.largest,w.peak);
      fflush(stderr);
    }
  dx_device_free(ctx,w.d); dx_device_free(ctx,w.d_out); dx_pinned_free(ctx,w.stage);
}

/* DEXB200_WINDOW=<bytes>, else the device's free memory over what a window needs per input byte */
static size_t window_size(const dx_tool *tool, dx_ctx *ctx)
{ const char *e = getenv("DEXB200_WINDOW");
  size_t win;
  if (e != NULL)
    win = (size_t) strtoull(e,NULL,10);
  else
    { size_t free = 0;
      if (dx_mem_info(ctx,&free,NULL,NULL) != DX_OK) die(ctx,DX_E_CUDA);
      win = (size_t) ((double) free / tool->expand);
    }
  return (win < MINWIN) ? MINWIN : win;
}

int dx_cli_main(const dx_tool *tool, int argc, char *argv[])
{ dx_opts o = { 0, 0, 0, 0, 0, 80 };
  int i, j, k;
  dx_ctx *ctx = NULL;
  size_t window = 0;

  Prog = tool->name;
  j = 1;
  for (i = 1; i < argc; i++)
    if (argv[i][0] == '-')
      { if (tool->has_width && argv[i][1] == 'w')                    /* ARG_NON_NEGATIVE */
          { char *eptr;
            o.width = (int) strtol(argv[i]+2,&eptr,10);
            if (*eptr != '\0' || argv[i][2] == '\0')
              { fprintf(stderr,"%s: -%c '%s' argument is not an integer\n",Prog,argv[i][1],argv[i]+2);
                exit (1);
              }
            if (o.width < 0)
              { fprintf(stderr,"%s: %s must be non-negative (%d)\n",Prog,"Line width",o.width);
                exit (1);
              }
            if (o.width == 0)      /* the reference loops forever on -w0 (undexta.c:265) */
              { fprintf(stderr,"%s: Line width must be positive (0)\n",Prog);
                exit (1);
              }
            continue;
          }
        for (k = 1; argv[i][k] != '\0'; k++)                          /* ARG_FLAGS */
          { if (strchr(tool->flags,argv[i][k]) == NULL)
              { fprintf(stderr,"%s: -%c is an illegal option\n",Prog,argv[i][k]);
                exit (1);
              }
            switch (argv[i][k])
              { case 'v': o.verbose = 1; break;
                case 'k': o.keep = 1; break;
                case 'i': o.pipe = 1; break;
                case 'U': o.upper = 1; break;
                case 'l': o.lossy = 1; break;
              }
          }
      }
    else
      argv[j++] = argv[i];
  argc = j;

  if ((o.pipe && argc > 1) || (!o.pipe && argc <= 1))
    { fprintf(stderr,"Usage: %s %s\n",Prog,tool->usage);
      fprintf(stderr,"\n");
      for (k = 0; k < 5 && tool->help[k] != NULL; k++)
        fprintf(stderr,"%s\n",tool->help[k]);
      exit (1);
    }
  if (o.pipe)
    { o.keep = 1; argc = 2; }

  for (i = 1; i < argc; i++)
    { char *src = NULL, *dst = NULL, *root;
      FILE *in, *out = NULL;
      uint8_t *h_in = NULL, *h_out = NULL, *d_in = NULL, *d_out = NULL;
      size_t n, m = 0;
      off_t fsize;
      int rc;

      if (o.pipe)
        { in = stdin; out = stdout;
          root = strdup("Standard Input");
        }
      else
        { src  = file_name(argv[i],tool->src_ext,tool->src_ext);
          dst  = file_name(argv[i],tool->src_ext,tool->dst_ext);
          root = root_name(argv[i],tool->src_ext);
          if ((in = fopen(src,"r")) == NULL)
            { fprintf(stderr,"%s: Cannot open %s for 'r'\n",Prog,src); exit (1); }
        }
      /* the device is opened once a source is: a missing file is reported the way the reference
         reports it, and no output file is created when there is no GPU to fill it */
      if (ctx == NULL)
        { int dev = 0;
          const char *e = getenv("DEXB200_DEVICE");
          if (e != NULL) dev = atoi(e);
          if (dx_open(dev,&ctx) != DX_OK) die(NULL,DX_E_NOGPU);
          window = window_size(tool,ctx);
        }
      if (!o.pipe && (out = fopen(dst,"w")) == NULL)
        { fprintf(stderr,"%s: Cannot open %s for 'w'\n",Prog,dst); exit (1); }
      if (o.verbose)
        { fprintf(stderr,"Processing '%s' ...\n",root); fflush(stderr); }

      { struct stat sb;                        /* a file larger than one window goes window by window */
        fsize = (!o.pipe && fstat(fileno(in),&sb) == 0 && S_ISREG(sb.st_mode)) ? sb.st_size : -1;
      }
      if (fsize < 0 || (size_t) fsize > window)
        { run_windows(tool,&o,ctx,in,out,window,fsize);
          goto written;
        }
      h_in = slurp(ctx,in,&n);
      d_in = (uint8_t *) dx_device_alloc(ctx,n + 64);
      if (d_in == NULL) die(ctx,DX_E_NOMEM);
      if ((rc = dx_h2d(ctx,d_in,h_in,n)) != DX_OK) die(ctx,rc);
      rc = tool->run(ctx,&o,d_in,n,&d_out,&m);
      if (rc == DX_E_NOMEM && n > 2*MINWIN && tool->stream != NULL)
        { /* the estimate of what a window needs was too low: half the file per window */
          dx_pinned_free(ctx,h_in); dx_device_free(ctx,d_in); dx_device_free(ctx,d_out);
          h_in = NULL; d_in = NULL; d_out = NULL;
          rewind(in);
          run_windows(tool,&o,ctx,in,out,n/2,fsize);
          goto written;
        }
      if (rc != DX_OK) die(ctx,rc);
      h_out = (uint8_t *) dx_pinned_alloc(ctx,m + 1);
      if (h_out == NULL) die(ctx,DX_E_NOMEM);
      if ((rc = dx_d2h(ctx,h_out,d_out,m)) != DX_OK) die(ctx,rc);
      if ((rc = dx_sync(ctx)) != DX_OK) die(ctx,rc);
      if (m > 0 && fwrite(h_out,1,m,out) != m)
        { fprintf(stderr,"%s: System error, write failed!\n",Prog); exit (2); }
written:

      /* the source is removed only after the output is completely written (SURVEY section 5) */
      if (!o.pipe)
        { fclose(in);
          if (fclose(out) != 0)
            { fprintf(stderr,"%s: System error, write failed!\n",Prog); exit (2); }
          if (!o.keep) unlink(src);
        }
      else
        fflush(out);
      dx_pinned_free(ctx,h_in); dx_pinned_free(ctx,h_out);
      dx_device_free(ctx,d_in); dx_device_free(ctx,d_out);
      free(src); free(dst); free(root);
      if (o.verbose)
        { fprintf(stderr,"Done\n"); fflush(stderr); }
    }
  dx_close(ctx);
  return 0;
}
