/* undexqv_mg -- undexqv of ONE .dexqv file on N GPUs of one node: .dexqv -> .quiva, the same bytes the
 * reference's undexqv writes (undexqv.c:99-208), the file cut into N byte ranges.
 *
 *     undexqv_mg [-vkU] -g<N> <path:dexqv> ...
 *
 * One process, one host thread per rank; rank r opens device r % (visible devices), so several ranks
 * may share a GPU.  Rank r takes the entries whose first byte lies in [r*n/N, (r+1)*n/N) and reads the
 * file from 4 KB in front of that cut to SLACK behind it (longer when the library asks for more:
 * DX_E_CAP, dx_needed_bytes).  Three library calls per rank (include/dexb200.h, dx_undexqv_range_*):
 *   1. dx_undexqv_range_dev       every rank at once: the range's entry candidates, decoded;
 *   2. dx_undexqv_range_chain     in rank order: the chain position and well number of the entry behind
 *                                 the previous range come in, those behind this range go out (host
 *                                 memory and a condition variable: a few scalars, no NCCL);
 *   3. dx_undexqv_range_text_dev  every rank at once: its text, written with pwrite at the sum of the
 *                                 text sizes of the ranks before it.
 * An image of the old layout or the other byte order, and a file smaller than N MB, are decoded by
 * rank 0 alone (dx_undexqv_dev).
 * Same file naming, flags, messages and exit codes as undexqv; the source is removed only after the
 * output is completely written.  Host code is plain C; every codec step runs on the GPUs.
 */
#define _GNU_SOURCE
#include <fcntl.h>
#include <pthread.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <strings.h>
#include <sys/stat.h>
#include <sys/time.h>
#include <unistd.h>
#include "dexb200.h"

#define MAXGPU   16
#define STAGE    ((size_t) 64 << 20)         /* pinned staging buffer per rank */
#define SLACK    ((size_t) 96 << 20)         /* read behind a rank's cut: the tails of its last entries */
#define BACK     4096                        /* read in front of it: what the range decode looks back at */
#define HEADMAX  ((size_t) 2 + 16384 + 100001)   /* key + coding header + prefix, at most */

static const char *Prog = "undexqv_mg";

typedef struct
  { int verbose, keep, upper, world, visible; } Opts;

typedef struct                               /* one file, shared by its ranks */
  { const Opts     *o;
    int             fd_in, fd_out;
    int64_t         fsize;
    uint8_t        *head;                    /* the file's first min(fsize, HEADMAX) bytes */
    size_t          head_n;
    pthread_mutex_t mu;
    pthread_cond_t  cv;
    int             chain_ready[MAXGPU+1], text_ready[MAXGPU+1];
    int64_t         cur[MAXGPU+1], tsize[MAXGPU+1];
    int32_t         well[MAXGPU+1];
  } Job;

typedef struct
  { int     rank;
    Job    *J;
    double  t_read, t_decode, t_relay, t_text, t_write;
    int64_t rbytes, wbytes;
  } Rank;

static double now(void)
{ struct timeval tv; gettimeofday(&tv,NULL); return tv.tv_sec + 1e-6*tv.tv_usec; }

static void die(dx_ctx *ctx, int rc)         /* undexqv's conventions (dxcli.c) */
{ if (rc == DX_E_TRUNC)
    { fprintf(stderr,"%s: System error, read failed!\n",Prog);
      exit (2);
    }
  fprintf(stderr,"%s: %s\n",Prog,ctx ? dx_strerror(ctx) : "cannot open a CUDA device (no CPU fallback)");
  exit (1);
}
#define DXC(call) do { int rc__ = (call); if (rc__ != DX_OK) die(ctx,rc__); } while (0)

static void read_at(int fd, uint8_t *dst, size_t len, int64_t at)
{ size_t have = 0;
  while (have < len)
    { ssize_t got = pread(fd,dst + have,len - have,at + (int64_t) have);
      if (got <= 0) { fprintf(stderr,"%s: System error, read failed!\n",Prog); exit (2); }
      have += (size_t) got;
    }
}

static void write_at(int fd, const uint8_t *src, size_t len, int64_t at)
{ if (len > 0 && pwrite(fd,src,len,at) != (ssize_t) len)
    { fprintf(stderr,"%s: System error, write failed!\n",Prog); exit (2); }
}

/* file bytes [from, to) -> device */
static void load(dx_ctx *ctx, int fd, uint8_t *stage, uint8_t *d_dst, int64_t from, int64_t to)
{ while (from < to)
    { size_t len = (size_t) (to - from) < STAGE ? (size_t) (to - from) : STAGE;
      read_at(fd,stage,len,from);
      DXC(dx_h2d(ctx,d_dst,stage,len));
      DXC(dx_sync(ctx));
      d_dst += len; from += (int64_t) len;
    }
}

/* device bytes -> file at `at` */
static void store(dx_ctx *ctx, int fd, uint8_t *stage, const uint8_t *d_src, size_t len, int64_t at)
{ for (size_t k = 0; k < len; k += STAGE)
    { size_t part = (len - k < STAGE) ? len - k : STAGE;
      DXC(dx_d2h(ctx,stage,d_src + k,part));
      DXC(dx_sync(ctx));
      write_at(fd,stage,part,at + (int64_t) k);
    }
}

static void *rank_main(void *arg)
{ Rank *R = (Rank *) arg;
  Job *J = R->J;
  const int W = J->o->world, r = R->rank;
  dx_ctx *ctx = NULL;
  { int rc = dx_open(r % J->o->visible,&ctx); if (rc != DX_OK) die(NULL,rc); }
  uint8_t *stage = (uint8_t *) dx_pinned_alloc(ctx,STAGE);
  if (stage == NULL) die(ctx,DX_E_NOMEM);
  double t0 = now();

  /* ---- 1. my bytes, my candidates decoded ------------------------------------------------------ */
  const int64_t n = J->fsize, a = n*r/W, b = n*(r+1)/W;
  const int64_t from = ((a > BACK) ? a - BACK : 0) & ~(int64_t) 15;
  int64_t to = (b + (int64_t) SLACK < n) ? b + (int64_t) SLACK : n;
  uint8_t *d_buf = NULL;
  int64_t first = 0, cur = 0, cur_out = 0;
  int32_t well = 0, well_out = 0;
  int chained = 0, rc;
  while (!chained)
    { dx_device_free(ctx,d_buf);
      if ((d_buf = (uint8_t *) dx_device_alloc(ctx,(size_t) (to - from) + 64)) == NULL) die(ctx,DX_E_NOMEM);
      load(ctx,J->fd_in,stage,d_buf,from,to);
      R->rbytes += to - from;
      R->t_read += now() - t0; t0 = now();
      rc = dx_undexqv_range_dev(ctx,J->head,J->head_n,d_buf,(size_t) (to - from),from,a,b,J->o->upper,&first);
      if (rc == DX_OK) rc = dx_sync(ctx);
      if (rc != DX_OK) die(ctx,rc);
      R->t_decode += now() - t0; t0 = now();

      /* ---- 2. the chain position of the range before me, then mine for the range behind me -------- */
      if (r == 0) { cur = first; well = 0; }
      else
        { pthread_mutex_lock(&J->mu);
          while (!J->chain_ready[r]) pthread_cond_wait(&J->cv,&J->mu);
          cur = J->cur[r]; well = J->well[r];
          pthread_mutex_unlock(&J->mu);
        }
      const double tw = now();
      rc = dx_undexqv_range_chain(ctx,cur,well,&cur_out,&well_out);
      if (rc == DX_E_CAP)                                  /* an entry's tail lies behind my buffer */
        { const int64_t need = (int64_t) dx_needed_bytes(ctx);
          if (to >= n) die(ctx,DX_E_TRUNC);                 /* the file ends inside an entry */
          to = (need > to && need < n) ? need : n;
          R->t_relay += now() - tw; t0 = now();
          continue;
        }
      if (rc != DX_OK) die(ctx,rc);
      chained = 1;
      R->t_relay += now() - tw; t0 = now();
    }
  if (r == W - 1 && cur_out != n) die(ctx,DX_E_TRUNC);
  pthread_mutex_lock(&J->mu);
  J->cur[r+1] = cur_out; J->well[r+1] = well_out; J->chain_ready[r+1] = 1;
  pthread_cond_broadcast(&J->cv);
  pthread_mutex_unlock(&J->mu);

  /* ---- 3. my text, at the sum of the text sizes before me ------------------------------------------ */
  size_t m = 0;
  uint8_t *d_out = NULL;
  rc = dx_undexqv_range_text_dev(ctx,NULL,0,&m);
  if (rc == DX_E_CAP)
    { m = dx_needed_bytes(ctx);
      if ((d_out = (uint8_t *) dx_device_alloc(ctx,m + 64)) == NULL) die(ctx,DX_E_NOMEM);
      rc = dx_undexqv_range_text_dev(ctx,d_out,m + 64,&m);
    }
  if (rc != DX_OK) die(ctx,rc);
  dx_device_free(ctx,d_buf);
  R->t_text = now() - t0;
  pthread_mutex_lock(&J->mu);
  J->tsize[r] = (int64_t) m; J->text_ready[r] = 1;
  pthread_cond_broadcast(&J->cv);
  int64_t off = 0;
  for (int q = 0; q < r; q++)
    { while (!J->text_ready[q]) pthread_cond_wait(&J->cv,&J->mu);
      off += J->tsize[q];
    }
  pthread_mutex_unlock(&J->mu);
  t0 = now();
  store(ctx,J->fd_out,stage,d_out,m,off);
  R->t_write = now() - t0;
  R->wbytes = (int64_t) m;
  dx_device_free(ctx,d_out);
  dx_pinned_free(ctx,stage);
  dx_close(ctx);
  return NULL;
}

/* the whole file on rank 0's device (dx_undexqv_dev), as undexqv decodes it */
static void decode_whole(Job *J)
{ dx_ctx *ctx = NULL;
  { int rc = dx_open(0,&ctx); if (rc != DX_OK) die(NULL,rc); }
  const size_t n = (size_t) J->fsize;
  uint8_t *stage = (uint8_t *) dx_pinned_alloc(ctx,STAGE);
  uint8_t *d_in = (uint8_t *) dx_device_alloc(ctx,n + 64), *d_out;
  size_t cap = 0, m = 0;
  if (stage == NULL || d_in == NULL) die(ctx,DX_E_NOMEM);
  load(ctx,J->fd_in,stage,d_in,0,(int64_t) n);
  DXC(dx_undexqv_size_dev(ctx,d_in,n,&cap));
  if ((d_out = (uint8_t *) dx_device_alloc(ctx,cap + 64)) == NULL) die(ctx,DX_E_NOMEM);
  DXC(dx_undexqv_dev(ctx,d_in,n,J->o->upper,d_out,cap + 64,&m,NULL,0,0));
  store(ctx,J->fd_out,stage,d_out,m,0);
  dx_device_free(ctx,d_in); dx_device_free(ctx,d_out); dx_pinned_free(ctx,stage);
  dx_close(ctx);
}

/* <dir>/<root><ext> from a command-line name, as dxcli.c (PathTo/Root/Catenate, DB.c:112-181) */
static char *file_name(const char *arg, const char *strip, const char *ext)
{ size_t la = strlen(arg), ls = strlen(strip);
  char *out = (char *) malloc(la + strlen(ext) + 16);
  const char *base = strrchr(arg,'/');
  size_t pre = 0;
  if (base == NULL)
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

int main(int argc, char *argv[])
{ Opts o = { 0, 0, 0, 0, 0 };
  int i, j = 1, k;
  for (i = 1; i < argc; i++)
    if (argv[i][0] == '-')
      { if (argv[i][1] == 'g') { o.world = atoi(argv[i]+2); continue; }
        for (k = 1; argv[i][k] != '\0'; k++)
          switch (argv[i][k])
            { case 'v': o.verbose = 1; break;
              case 'k': o.keep = 1; break;
              case 'U': o.upper = 1; break;
              default:
                fprintf(stderr,"%s: -%c is an illegal option\n",Prog,argv[i][k]); exit (1);
            }
      }
    else
      argv[j++] = argv[i];
  argc = j;
  if (argc <= 1 || o.world < 1 || o.world > MAXGPU)
    { fprintf(stderr,"Usage: %s [-vkU] -g<gpus(1..%d)> <path:dexqv> ...\n\n",Prog,MAXGPU);
      fprintf(stderr,"      -k: do *not* remove the .dexqv file on completion.\n");
      fprintf(stderr,"      -U: use uppercase letters (default is lower case).\n");
      fprintf(stderr,"      -g: decode each file on this many GPUs (rank r on device r %% visible devices).\n");
      exit (1);
    }
  for (i = 1; i < argc; i++)
    { char *src = file_name(argv[i],".dexqv",".dexqv"), *dst = file_name(argv[i],".dexqv",".quiva");
      char *root = root_name(argv[i],".dexqv");
      struct stat sb;
      Job J;
      Rank R[MAXGPU];
      pthread_t th[MAXGPU];
      int fd_in = open(src,O_RDONLY);
      double t0 = now();
      if (fd_in < 0 || fstat(fd_in,&sb) != 0)
        { fprintf(stderr,"%s: Cannot open %s for 'r'\n",Prog,src); exit (1); }
      if (o.visible == 0)                                  /* the devices are counted once a source is open */
        { dx_ctx *probe = NULL;
          while (o.visible < o.world && dx_open(o.visible,&probe) == DX_OK) { dx_close(probe); o.visible++; }
          if (o.visible == 0) die(NULL,DX_E_NOGPU);
        }
      memset(&J,0,sizeof(J));
      J.o = &o; J.fd_in = fd_in; J.fsize = (int64_t) sb.st_size;
      J.head_n = ((size_t) sb.st_size < HEADMAX) ? (size_t) sb.st_size : HEADMAX;
      J.head = (uint8_t *) malloc(J.head_n + 1);
      read_at(fd_in,J.head,J.head_n,0);
      if ((J.fd_out = open(dst,O_WRONLY|O_CREAT|O_TRUNC,0644)) < 0)
        { fprintf(stderr,"%s: Cannot open %s for 'w'\n",Prog,dst); exit (1); }
      if (o.verbose) { fprintf(stderr,"Processing '%s' ...\n",root); fflush(stderr); }
      pthread_mutex_init(&J.mu,NULL); pthread_cond_init(&J.cv,NULL);
      /* rank 0 alone: not the native 0x55aa layout (the old layout, the other byte order), or too small */
      const int whole = !(J.head_n >= 2 && J.head[0] == 0xaa && J.head[1] == 0x55) || J.fsize < (int64_t) o.world << 20;
      if (whole)
        { if (o.verbose)
            { fprintf(stderr,"  %s: rank 0 decodes the file alone\n",
                      J.fsize < (int64_t) o.world << 20 ? "smaller than 1 MB per GPU" : "old layout or other byte order");
              fflush(stderr);
            }
          decode_whole(&J);
        }
      else
        { for (k = 0; k < o.world; k++)
            { memset(&R[k],0,sizeof(Rank));
              R[k].rank = k; R[k].J = &J;
              if (pthread_create(&th[k],NULL,rank_main,&R[k]) != 0) { fprintf(stderr,"%s: pthread_create failed\n",Prog); exit (1); }
            }
          for (k = 0; k < o.world; k++) pthread_join(th[k],NULL);
        }
      close(fd_in);
      if (close(J.fd_out) != 0) { fprintf(stderr,"%s: System error, write failed!\n",Prog); exit (2); }
      if (o.verbose && !whole)
        { double tr = 0, td = 0, tc = 0, tt = 0, tw = 0; int64_t rb = 0, wb = 0;
          for (k = 0; k < o.world; k++)
            { if (R[k].t_read > tr)   tr = R[k].t_read;
              if (R[k].t_decode > td) td = R[k].t_decode;
              if (R[k].t_relay > tc)  tc = R[k].t_relay;
              if (R[k].t_text > tt)   tt = R[k].t_text;
              if (R[k].t_write > tw)  tw = R[k].t_write;
              rb += R[k].rbytes; wb += R[k].wbytes;
            }
          fprintf(stderr,"  %lld bytes on %d GPUs (%d devices) -> %lld bytes; max over ranks: read+H2D %.3f s, "
                         "decode %.3f s, walk+relay %.3f s, text %.3f s, D2H+write %.3f s; wall %.3f s\n",
                  (long long) J.fsize,o.world,o.visible,(long long) wb,tr,td,tc,tt,tw,now() - t0);
          for (k = 0; k < o.world; k++)
            fprintf(stderr,"  rank %d (device %d): read %lld bytes, wrote %lld; read+H2D %.3f s, decode %.3f s, "
                           "walk+relay %.3f s, text %.3f s, D2H+write %.3f s\n",k,k % o.visible,(long long) R[k].rbytes,
                    (long long) R[k].wbytes,R[k].t_read,R[k].t_decode,R[k].t_relay,R[k].t_text,R[k].t_write);
        }
      /* the source is removed only after the output is completely written */
      if (!o.keep) unlink(src);
      pthread_mutex_destroy(&J.mu); pthread_cond_destroy(&J.cv);
      free(J.head); free(src); free(dst); free(root);
      if (o.verbose) { fprintf(stderr,"Done\n"); fflush(stderr); }
    }
  return 0;
}
