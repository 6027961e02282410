// dx_api.cpp -- the C ABI of libdexb200.so (include/dexb200.h): context, device scratch arena,
// and the host-side orchestration of the kernels.  The host does only what the reference does
// once per file (prefix, coding header, code-length assignment) or what costs O(#entries)
// integer work (header text lengths, chain verification); every per-symbol loop is a kernel.
//
// There is no CPU implementation of the codecs in this library: without a CUDA device dx_open
// fails with DX_E_NOGPU and nothing else can be called.

#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include <algorithm>
#include <chrono>
#include <new>
#include <unordered_map>
#include "dx_internal.h"
#include "dx_chain.h"

// wall-clock marks of the host phases of a call, printed with DEXB200_DEBUG set
struct DxPhases
{ bool on; std::chrono::steady_clock::time_point t0; char buf[512]; size_t len;
  explicit DxPhases(const dx_ctx *ctx) : on(ctx->route[DXR_DEBUG] != 0), len(0) { buf[0] = 0; t0 = std::chrono::steady_clock::now(); }
  void mark(const char *what)
  { if (!on) return;
    auto t1 = std::chrono::steady_clock::now();
    len += (size_t) snprintf(buf+len,sizeof(buf)-len," %s %.3f",what,
                             std::chrono::duration<double,std::milli>(t1-t0).count());
    if (len >= sizeof(buf)) len = sizeof(buf)-1;
    t0 = t1;
  }
  void report(const char *call) { if (on) fprintf(stderr,"[dexb200 debug] %s host phases (ms):%s\n",call,buf); }
};

// ================================================================================================
//  errors, context, arena
// ================================================================================================

// every DX_E_CAP failure clears the size kept for dx_needed_bytes, so a caller never reallocates from
// what an earlier call needed; dx_fail_cap then sets it when the call knows its size
int dx_fail(dx_ctx *ctx, int code, const char *fmt, ...)
{ if (ctx != NULL)
    { if (code == DX_E_CAP) ctx->need_bytes = 0;
      va_list ap;
      va_start(ap,fmt);
      vsnprintf(ctx->err,sizeof(ctx->err),fmt,ap);
      va_end(ap);
    }
  return code;
}

// the output buffer is too small: the size the call needs is kept for dx_needed_bytes
int dx_fail_cap(dx_ctx *ctx, size_t need, size_t cap)
{ dx_fail(ctx,DX_E_CAP,"output needs %zu bytes, buffer has %zu",need,cap);
  ctx->need_bytes = need;
  return DX_E_CAP;
}

int dx_cuda_fail(dx_ctx *ctx, cudaError_t e, const char *what)
{ return dx_fail(ctx,DX_E_CUDA,"CUDA error %d (%s) in %s",(int) e,cudaGetErrorString(e),what); }

static size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

void dx_arena_reset(dx_ctx *ctx)
{ if (ctx->nblk > 1)
    { // the last call spilled over: consolidate into one block big enough for all of it
      size_t total = 0;
      for (int i = 0; i < ctx->nblk; i++)
        { total += ctx->blk[i].cap;
          cudaFree(ctx->blk[i].p);
        }
      ctx->nblk = 0;
      uint8_t *p = NULL;
      total = round_up(total + total/4,(size_t) 1 << 20);
      if (cudaMalloc((void **) &p,total) == cudaSuccess)
        { ctx->blk[0].p = p; ctx->blk[0].cap = total; ctx->blk[0].top = 0; ctx->nblk = 1; }
      else
        cudaGetLastError();
    }
  for (int i = 0; i < ctx->nblk; i++)
    ctx->blk[i].top = 0;
  ctx->hpin_top = 0;
  ctx->qv_range_live = 0;                               // its scratch is gone
}

// Pinned host scratch.  Pointers stay valid until the next dx_arena_reset: when the block is too
// small a bigger one REPLACES it only if nothing has been handed out yet, else a one-off
// allocation is chained behind it (freed at the next reset).
struct DxPinExtra { void *p; DxPinExtra *next; };

void *dx_hpin_get(dx_ctx *ctx, size_t bytes)
{ bytes = round_up(bytes > 0 ? bytes : 1,64);
  if (ctx->hpin_top == 0)
    { while (ctx->hpin_extra)
        { DxPinExtra *e = (DxPinExtra *) ctx->hpin_extra; ctx->hpin_extra = e->next; cudaFreeHost(e->p); free(e); }
      if (ctx->hpin_cap < bytes || ctx->hpin_cap < ctx->hpin_want)
        { if (ctx->hpin) cudaFreeHost(ctx->hpin);
          ctx->hpin = NULL; ctx->hpin_cap = 0;
          size_t want = round_up((bytes > ctx->hpin_want ? bytes : ctx->hpin_want)*2,(size_t) 1 << 20);
          if (cudaMallocHost((void **) &ctx->hpin,want) != cudaSuccess)
            { cudaGetLastError(); dx_fail(ctx,DX_E_NOMEM,"pinned host allocation of %zu bytes failed",want); return NULL; }
          ctx->hpin_cap = want;
        }
    }
  if (ctx->hpin_top + bytes <= ctx->hpin_cap)
    { void *p = ctx->hpin + ctx->hpin_top; ctx->hpin_top += bytes; return p; }
  DxPinExtra *e = (DxPinExtra *) malloc(sizeof(DxPinExtra));
  if (e == NULL || cudaMallocHost(&e->p,bytes) != cudaSuccess)
    { cudaGetLastError(); free(e); dx_fail(ctx,DX_E_NOMEM,"pinned host allocation of %zu bytes failed",bytes); return NULL; }
  e->next = (DxPinExtra *) ctx->hpin_extra; ctx->hpin_extra = e;
  ctx->hpin_top += bytes;                               // past the block: every later request is a one-off too
  if (ctx->hpin_top > ctx->hpin_want) ctx->hpin_want = ctx->hpin_top;
  return e->p;
}

void *dx_arena_get(dx_ctx *ctx, size_t bytes)
{ bytes = round_up(bytes > 0 ? bytes : 1,256);
  for (int i = 0; i < ctx->nblk; i++)
    if (ctx->blk[i].top + bytes <= ctx->blk[i].cap)
      { void *p = ctx->blk[i].p + ctx->blk[i].top;
        ctx->blk[i].top += bytes;
        return p;
      }
  if (ctx->nblk >= 32)
    { dx_fail(ctx,DX_E_NOMEM,"scratch arena exhausted (32 blocks)");
      return NULL;
    }
  size_t cap = round_up(bytes > ((size_t) 32 << 20) ? bytes : ((size_t) 32 << 20),(size_t) 1 << 20);
  if (ctx->route[DXR_ARENA_CAP] > 0)
    { size_t have = 0;
      for (int i = 0; i < ctx->nblk; i++) have += ctx->blk[i].cap;
      if (have + cap > (size_t) ctx->route[DXR_ARENA_CAP])
        { dx_fail(ctx,DX_E_NOMEM,"scratch arena capped at %lld bytes (arena_cap)",(long long) ctx->route[DXR_ARENA_CAP]);
          return NULL;
        }
    }
  uint8_t *p = NULL;
  cudaError_t e = cudaMalloc((void **) &p,cap);
  if (e != cudaSuccess)
    { cudaGetLastError();                               // not left behind for the next launch check
      dx_cuda_fail(ctx,e,"cudaMalloc(scratch)");
      return NULL;
    }
  DxBlock &b = ctx->blk[ctx->nblk++];
  b.p = p; b.cap = cap; b.top = bytes;
  return p;
}

int dx_arena_reserve(dx_ctx *ctx, size_t bytes)
{ void *p = dx_arena_get(ctx,bytes);
  if (p == NULL) return DX_E_NOMEM;
  dx_arena_reset(ctx);
  return DX_OK;
}

// ---- per-kernel event timing -------------------------------------------------------------------

struct DxProfRec { const char *name; cudaEvent_t a, b; };
struct DxProf : std::vector<DxProfRec>
{ std::vector<cudaEvent_t> pool;                    // events of earlier reports, reused
  cudaEvent_t get()
  { cudaEvent_t e;
    if (!pool.empty()) { e = pool.back(); pool.pop_back(); }
    else cudaEventCreate(&e);
    return e;
  }
};

void dx_prof_begin(dx_ctx *ctx)
{ DxProf *pv = (DxProf *) ctx->prof;
  DxProfRec r; r.name = NULL;
  r.a = pv->get(); r.b = pv->get();
  cudaEventRecord(r.a,ctx->stream);
  pv->push_back(r);
}

void dx_prof_end(dx_ctx *ctx, const char *what)
{ DxProf *pv = (DxProf *) ctx->prof;
  if (pv->empty() || pv->back().name != NULL) return;
  pv->back().name = what;
  cudaEventRecord(pv->back().b,ctx->stream);
}

extern "C" int dx_profile(dx_ctx *ctx, int enable)
{ if (ctx == NULL) return DX_E_ARG;
  if (ctx->prof == NULL) ctx->prof = new DxProf();
  ctx->prof_on = enable ? 1 : 0;
  return DX_OK;
}

extern "C" int dx_profile_report(dx_ctx *ctx, char *buf, size_t cap)
{ if (ctx == NULL || buf == NULL || cap == 0) return DX_E_ARG;
  buf[0] = '\0';
  if (ctx->prof == NULL) return DX_OK;
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  DxProf *pv = (DxProf *) ctx->prof;
  struct Acc { const char *name; int calls; double ms; };
  std::vector<Acc> acc;
  for (DxProfRec &r : *pv)
    { float ms = 0;
      if (r.name != NULL && cudaEventElapsedTime(&ms,r.a,r.b) == cudaSuccess)
        { size_t k = 0;
          while (k < acc.size() && strcmp(acc[k].name,r.name) != 0) k++;
          if (k == acc.size()) acc.push_back(Acc{r.name,0,0.0});
          acc[k].calls += 1; acc[k].ms += ms;
        }
      pv->pool.push_back(r.a); pv->pool.push_back(r.b);
    }
  pv->clear();
  size_t at = 0;
  for (const Acc &a : acc)
    { int w = snprintf(buf+at,cap-at,"%s %d %.6f\n",a.name,a.calls,a.ms);
      if (w < 0 || (size_t) w >= cap-at) return dx_fail(ctx,DX_E_CAP,"profile report needs more than %zu bytes",cap);
      at += (size_t) w;
    }
  return DX_OK;
}

extern "C" int dx_open(int device, dx_ctx **out)
{ if (out == NULL) return DX_E_ARG;
  *out = NULL;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    { cudaGetLastError();
      return DX_E_NOGPU;
    }
  if (device < 0 || device >= ndev) return DX_E_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return DX_E_CUDA;
  dx_ctx *ctx = (dx_ctx *) calloc(1,sizeof(dx_ctx));
  if (ctx == NULL) return DX_E_NOMEM;
  ctx->device = device;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop,device) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->stream,cudaStreamNonBlocking) != cudaSuccess)
    { free(ctx);
      return DX_E_CUDA;
    }
  ctx->sm_count = prop.multiProcessorCount;
  ctx->route[DXR_DEBUG] = (getenv("DEXB200_DEBUG") != NULL);      // read once, here; never in a call
  { const char *cap = getenv("DEXB200_ARENA_CAP");                  // tests: out-of-memory in a subprocess
    if (cap != NULL) ctx->route[DXR_ARENA_CAP] = strtoll(cap,NULL,10);
  }
  *out = ctx;
  return DX_OK;
}

static void qv_range_free(dx_ctx *ctx);

extern "C" void dx_close(dx_ctx *ctx)
{ if (ctx == NULL) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (int i = 0; i < ctx->nblk; i++) cudaFree(ctx->blk[i].p);
  if (ctx->io_in)    cudaFree(ctx->io_in);
  if (ctx->io_out)   cudaFree(ctx->io_out);
  if (ctx->qv_store) cudaFree(ctx->qv_store);
  if (ctx->last_index) delete (std::vector<dx_index_row> *) ctx->last_index;
  delete (std::unordered_map<void *,size_t> *) ctx->dev_blocks;
  qv_range_free(ctx);
  if (ctx->hpin)     cudaFreeHost(ctx->hpin);
  while (ctx->hpin_extra)
    { DxPinExtra *e = (DxPinExtra *) ctx->hpin_extra; ctx->hpin_extra = e->next; cudaFreeHost(e->p); free(e); }
  if (ctx->prof)
    { char tmp[16]; ctx->prof_on = 0; dx_profile_report(ctx,tmp,sizeof(tmp));
      for (cudaEvent_t e : ((DxProf *) ctx->prof)->pool) cudaEventDestroy(e);
      delete (DxProf *) ctx->prof;
    }
  for (int i = 0; i < ctx->npev; i++) cudaEventDestroy(ctx->pev[i]);
  if (ctx->cs_in)  cudaStreamDestroy(ctx->cs_in);
  if (ctx->cs_out) cudaStreamDestroy(ctx->cs_out);
  cudaStreamDestroy(ctx->stream);
  free(ctx);
}

extern "C" const char *dx_strerror(const dx_ctx *ctx) { return ctx ? ctx->err : "no context"; }
extern "C" int64_t     dx_error_line(const dx_ctx *ctx) { return ctx ? ctx->err_line : 0; }
extern "C" size_t      dx_needed_bytes(const dx_ctx *ctx) { return ctx ? ctx->need_bytes : 0; }
extern "C" void       *dx_stream(dx_ctx *ctx) { return ctx ? (void *) ctx->stream : NULL; }

extern "C" int dx_route(dx_ctx *ctx, const char *name, int64_t value)
{ static const char *names[DXR_COUNT] = { "no_fast", "no_spec", "exact_index", "exact_pack", "pack2", "two_pass",
                                          "chain_scan", "decoder", "lane_max_rlen", "lane_min_entries", "debug",
                                          "serial_io", "pipe_chunk", "no_direct", "index_bulk", "hist_mode",
                                          "arena_cap" };
  if (ctx == NULL || name == NULL) return DX_E_ARG;
  if (strcmp(name,"default") == 0)
    { const int64_t dbg = ctx->route[DXR_DEBUG], cap = ctx->route[DXR_ARENA_CAP];
      memset(ctx->route,0,sizeof(ctx->route));
      ctx->route[DXR_DEBUG] = dbg;
      ctx->route[DXR_ARENA_CAP] = cap;
      return DX_OK;
    }
  for (int k = 0; k < DXR_COUNT; k++)
    if (strcmp(name,names[k]) == 0) { ctx->route[k] = value; return DX_OK; }
  return dx_fail(ctx,DX_E_ARG,"dx_route: unknown route '%s'",name);
}

extern "C" int dx_keep_index(dx_ctx *ctx, int keep)
{ if (ctx == NULL) return DX_E_ARG;
  ctx->keep_index = keep;
  if (ctx->last_index == NULL) ctx->last_index = new std::vector<dx_index_row>();
  return DX_OK;
}

extern "C" int dx_last_index(dx_ctx *ctx, dx_index_row *rows, int64_t max, int64_t *count)
{ if (ctx == NULL || count == NULL) return DX_E_ARG;
  std::vector<dx_index_row> *v = (std::vector<dx_index_row> *) ctx->last_index;
  *count = v ? (int64_t) v->size() : 0;
  if (v && rows)
    for (int64_t i = 0; i < *count && i < max; i++) rows[i] = (*v)[(size_t) i];
  return DX_OK;
}

extern "C" int dx_sync(dx_ctx *ctx)
{ DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  return DX_OK;
}

extern "C" uint64_t dx_launch_count(dx_ctx *ctx, int reset)
{ uint64_t v = ctx->launches;
  if (reset) ctx->launches = 0;
  return v;
}

extern "C" void *dx_device_alloc(dx_ctx *ctx, size_t bytes)
{ void *p = NULL;
  cudaSetDevice(ctx->device);
  const size_t sz = round_up(bytes + 64,256);
  cudaError_t e = cudaMalloc(&p,sz);
  if (e != cudaSuccess) { cudaGetLastError(); dx_cuda_fail(ctx,e,"cudaMalloc"); return NULL; }
  if (ctx->dev_blocks == NULL) ctx->dev_blocks = new std::unordered_map<void *,size_t>();
  (*(std::unordered_map<void *,size_t> *) ctx->dev_blocks)[p] = sz;
  return p;
}
extern "C" void dx_device_free(dx_ctx *ctx, void *p)
{ if (p == NULL) return;
  if (ctx != NULL && ctx->dev_blocks != NULL) ((std::unordered_map<void *,size_t> *) ctx->dev_blocks)->erase(p);
  cudaFree(p);
}

extern "C" int dx_mem_info(dx_ctx *ctx, size_t *free_bytes, size_t *total_bytes, size_t *held)
{ if (ctx == NULL) return DX_E_ARG;
  cudaSetDevice(ctx->device);
  size_t f = 0, t = 0;
  DX_CUDA(ctx,cudaMemGetInfo(&f,&t));
  size_t h = ctx->io_in_cap + ctx->io_out_cap + ctx->qv_store_cap;
  for (int i = 0; i < ctx->nblk; i++) h += ctx->blk[i].cap;
  if (ctx->dev_blocks != NULL)
    for (const auto &b : *(std::unordered_map<void *,size_t> *) ctx->dev_blocks) h += b.second;
  if (free_bytes)  *free_bytes = f;
  if (total_bytes) *total_bytes = t;
  if (held)        *held = h;
  return DX_OK;
}

extern "C" int dx_set_origin(dx_ctx *ctx, int64_t line0, int64_t entry0)
{ if (ctx == NULL || line0 < 0 || entry0 < 0) return DX_E_ARG;
  ctx->origin_line = line0; ctx->origin_entry = entry0;
  return DX_OK;
}

extern "C" int64_t dx_last_entries(const dx_ctx *ctx) { return ctx ? ctx->last_entries : 0; }

extern "C" void *dx_pinned_alloc(dx_ctx *ctx, size_t bytes)
{ void *p = NULL;
  cudaError_t e = cudaHostAlloc(&p,bytes > 0 ? bytes : 1,cudaHostAllocDefault);
  if (e != cudaSuccess) { dx_cuda_fail(ctx,e,"cudaHostAlloc"); return NULL; }
  return p;
}
extern "C" void dx_pinned_free(dx_ctx *ctx, void *p) { (void) ctx; if (p) cudaFreeHost(p); }

extern "C" int dx_h2d(dx_ctx *ctx, void *d, const void *h, size_t n)
{ DX_CUDA(ctx,cudaMemcpyAsync(d,h,n,cudaMemcpyHostToDevice,ctx->stream)); return DX_OK; }
extern "C" int dx_d2d(dx_ctx *ctx, void *d_dst, const void *d_src, size_t n)
{ if (ctx == NULL) return DX_E_ARG;
  cudaSetDevice(ctx->device);
  if (n > 0) DX_CUDA(ctx,cudaMemcpyAsync(d_dst,d_src,n,cudaMemcpyDeviceToDevice,ctx->stream));
  return DX_OK;
}
extern "C" int dx_d2h(dx_ctx *ctx, void *h, const void *d, size_t n)
{ DX_CUDA(ctx,cudaMemcpyAsync(h,d,n,cudaMemcpyDeviceToHost,ctx->stream)); return DX_OK; }

// ---- small helpers ---------------------------------------------------------------------------

static int check_buf(dx_ctx *ctx, const void *p, const char *what)
{ if (p == NULL) return dx_fail(ctx,DX_E_ARG,"%s is NULL",what);
  if (((uintptr_t) p & 15) != 0)
    return dx_fail(ctx,DX_E_ARG,"%s must be 16-byte aligned device memory",what);
  return DX_OK;
}

// copy [at, at+len) of a device image to the host (synchronous)
static int peek(dx_ctx *ctx, const uint8_t *d, size_t n, size_t at, size_t len, std::vector<uint8_t> &h)
{ if (at > n) at = n;
  if (at + len > n) len = n - at;
  h.resize(len);
  if (len == 0) return DX_OK;
  DX_CUDA(ctx,cudaMemcpyAsync(h.data(),d+at,len,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  return DX_OK;
}

template <class T>
static int download(dx_ctx *ctx, const T *d, size_t count, std::vector<T> &h)
{ h.resize(count);
  if (count == 0) return DX_OK;
  DX_CUDA(ctx,cudaMemcpyAsync(h.data(),d,count*sizeof(T),cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  return DX_OK;
}

template <class T>
static int upload(dx_ctx *ctx, T *d, const T *h, size_t count)
{ if (count == 0) return DX_OK;
  DX_CUDA(ctx,cudaMemcpyAsync(d,h,count*sizeof(T),cudaMemcpyHostToDevice,ctx->stream));
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));     // h may be a temporary
  return DX_OK;
}

static int ndigits(int32_t v)          // characters printf("%d") produces
{ int n = (v < 0);
  uint32_t u = (v < 0) ? (uint32_t) (-(int64_t) v) : (uint32_t) v;
  do { n++; u /= 10; } while (u);
  return n;
}

static int ensure_io(dx_ctx *ctx, uint8_t **buf, size_t *cap, size_t need)
{ need = round_up(need + 64,256);
  if (*cap >= need) return DX_OK;
  if (*buf) cudaFree(*buf);
  *buf = NULL; *cap = 0;
  if (cudaMalloc((void **) buf,need) != cudaSuccess)
    { *buf = NULL; cudaGetLastError();
      return dx_fail(ctx,DX_E_NOMEM,"device allocation of %zu bytes (staging) failed",need);
    }
  *cap = need;
  return DX_OK;
}

// ================================================================================================
//  Chain of entries in a compressed image (.dexta / .dexar / .dexqv)
//
//  None of the three formats stores entry lengths; the reference finds entry k+1 only by
//  finishing entry k.  Here: every offset whose bytes look like an entry's fixed fields is a
//  CANDIDATE (dx_frame.cu); all candidates are walked in parallel to find where they would
//  end; then the host accepts a candidate only if the previous accepted entry ends exactly at
//  its well-delta bytes.  Exactness never depends on the candidate filter: a true entry the
//  filter missed is walked on its own (slow path), a false candidate is never reached.
// ================================================================================================

struct ChainEntry
{ int64_t start;        // first well-delta byte
  int64_t q;            // first field byte
  int64_t end;          // first byte after the entry
  int64_t cand;         // candidate index, or -1 when found by the slow path
  int32_t well;         // absolute well number
  uint8_t field[16];
};

typedef int (*WalkOne)(dx_ctx *ctx, void *user, int64_t q, int64_t *end, int64_t *slot);

static int resolve_chain(dx_ctx *ctx, const uint8_t *d_in, size_t n, size_t first, int fieldbytes,
                         const std::vector<int64_t> &q, const std::vector<int64_t> &end,
                         const std::vector<CandInfo> &info, WalkOne walk_one, void *user,
                         std::vector<ChainEntry> &chain)
{ int64_t cur = (int64_t) first;
  int32_t well = 0;
  size_t  i = 0;
  const size_t nc = q.size();
  chain.clear();
  std::vector<uint8_t> win;
  while (cur < (int64_t) n)
    { while (i < nc && q[i] - 1 < cur) i++;                  // candidates inside accepted entries
      // the entry at cur has its fields right after the run of 0xff bytes that starts at cur
      // and the one byte that ends it: a candidate is that entry iff its q is exactly there
      while (i < nc && info[i].last == 0xff && q[i] - 1 - cur <= info[i].ffrun)
        i++;                                                  // candidate inside the 0xff run
      bool ok = false;
      if (i < nc && end[i] >= 0)
        { const int64_t gap = q[i] - 1 - cur;                // must be all 0xff, then last != 0xff
          ok = (gap <= info[i].ffrun && info[i].last != 0xff);
        }
      ChainEntry ce;
      if (ok)
        { ce.start = cur; ce.q = q[i]; ce.end = end[i]; ce.cand = (int64_t) i;
          well += 255 * (int32_t) (q[i] - 1 - cur) + info[i].last;
          memcpy(ce.field,info[i].field,16);
          i++;
        }
      else
        { // slow path: read the header bytes at cur and walk this one entry by itself
          int64_t p = cur;
          int32_t add = 0;
          uint8_t byte = 0xff;
          while (byte == 0xff)
            { int rc = peek(ctx,d_in,n,(size_t) p,4096,win);
              if (rc != DX_OK) return rc;
              if (win.empty()) return dx_fail(ctx,DX_E_TRUNC,"compressed image ends inside an entry header");
              size_t k = 0;
              while (k < win.size() && win[k] == 0xff) { add += 255; k++; }
              p += (int64_t) k;
              if (k < win.size()) { byte = win[k]; add += byte; p += 1; }
            }
          int rc = peek(ctx,d_in,n,(size_t) p,16,win);
          if (rc != DX_OK) return rc;
          if ((int) win.size() < fieldbytes)
            return dx_fail(ctx,DX_E_TRUNC,"compressed image ends inside an entry header");
          memset(ce.field,0,16);
          memcpy(ce.field,win.data(),(size_t) fieldbytes);
          ce.start = cur; ce.q = p; ce.cand = -1;
          int64_t e = -1, slot = -1;
          rc = walk_one(ctx,user,p,&e,&slot);
          if (rc != DX_OK) return rc;
          ce.end = e;
          ce.cand = -2 - slot;                                // slot in the walker's side table
          well += add;
        }
      if (ce.end < 0 || ce.end > (int64_t) n || ce.end <= cur)
        return dx_fail(ctx,DX_E_TRUNC,"compressed image ends inside an entry (offset %lld)",
                       (long long) cur);
      ce.well = well;
      chain.push_back(ce);
      cur = ce.end;
    }
  return DX_OK;
}

static inline int32_t le32(const uint8_t *p)
{ return (int32_t) ((uint32_t) p[0] | ((uint32_t) p[1] << 8) | ((uint32_t) p[2] << 16) | ((uint32_t) p[3] << 24)); }

// ================================================================================================
//  2-bit codec
// ================================================================================================

struct PkWalkUser { int fieldbytes; const uint8_t *d_in; size_t n; };

static int pk_walk_one(dx_ctx *ctx, void *user, int64_t q, int64_t *end, int64_t *slot)
{ PkWalkUser *u = (PkWalkUser *) user;
  std::vector<uint8_t> f;
  int rc = peek(ctx,u->d_in,u->n,(size_t) q,(size_t) u->fieldbytes,f);
  if (rc != DX_OK) return rc;
  *slot = 0;
  if ((int) f.size() < u->fieldbytes) { *end = -1; return DX_OK; }
  const int64_t rlen = (int64_t) le32(f.data()+4) - le32(f.data());
  if (rlen < 0) return dx_fail(ctx,DX_E_FORMAT,"negative read length in entry header");
  *end = q + u->fieldbytes + ((rlen + 3) >> 2);
  return DX_OK;
}

static int dexta_impl(dx_ctx *ctx, int kind, const uint8_t *d_text, size_t n, int32_t lwell_in, int with_header,
                      uint8_t *d_out, size_t cap, size_t *out_len, int32_t *last_well, bool exact, bool *redo);

extern "C" int dx_dexta_part_dev(dx_ctx *ctx, int kind, const uint8_t *d_text, size_t n, int32_t lwell_in,
                                 int with_header, uint8_t *d_out, size_t cap, size_t *out_len, int32_t *last_well)
{ if (ctx == NULL) return DX_E_ARG;
  // first the vectorised kernels, which take the symbol counts from the line lattice and verify them
  // while packing; a file whose lines do not form the lattice is redone with the exact counts
  bool redo = false;
  int rc = dexta_impl(ctx,kind,d_text,n,lwell_in,with_header,d_out,cap,out_len,last_well,
                      ctx->route[DXR_EXACT_PACK] != 0,&redo);
  if (rc == DX_OK && redo) rc = dexta_impl(ctx,kind,d_text,n,lwell_in,with_header,d_out,cap,out_len,last_well,true,&redo);
  return rc;
}

extern "C" int dx_dexta_dev(dx_ctx *ctx, int kind, const uint8_t *d_text, size_t n,
                            uint8_t *d_out, size_t cap, size_t *out_len)
{ return dx_dexta_part_dev(ctx,kind,d_text,n,0,1,d_out,cap,out_len,NULL); }

static int dexta_impl(dx_ctx *ctx, int kind, const uint8_t *d_text, size_t n, int32_t lwell_in, int with_header,
                      uint8_t *d_out, size_t cap, size_t *out_len, int32_t *last_well, bool exact, bool *redo)
{ *redo = false;
  if (ctx == NULL || out_len == NULL || (kind != DX_FASTA && kind != DX_ARROW)) return DX_E_ARG;
  *out_len = 0;
  ctx->err_line = 0;
  ctx->last_entries = 0;
  int rc;
  if ((rc = check_buf(ctx,d_text,"text")) != DX_OK) return rc;
  if (d_out == NULL) return dx_fail(ctx,DX_E_ARG,"output is NULL");
  if (n == 0) return dx_fail(ctx,DX_E_FORMAT,"empty input");
  cudaSetDevice(ctx->device);
  dx_arena_reset(ctx);

  // first header line: endian key + prefix (dexta.c:108-129); a later part only has to start at a header
  std::vector<uint8_t> head;
  int32_t plen = 0;
  size_t  hbytes = 0;
  if ((rc = peek(ctx,d_text,n,0,with_header ? 100000 : 1,head)) != DX_OK) return rc;
  if (with_header)
    { const uint8_t *nl = (const uint8_t *) memchr(head.data(),'\n',head.size());
      if (nl == NULL || nl - head.data() > 99998)
        { ctx->err_line = 1;
          return dx_fail(ctx,DX_E_TOOLONG,"Line 1: %s line is too long (> 99998 chars)",
                         kind == DX_FASTA ? "Fasta" : "Arrow");
        }
      if (head[0] != '>')
        { ctx->err_line = 1;
          return dx_fail(ctx,DX_E_FORMAT,"Line 1: First header in %s file is missing",
                         kind == DX_FASTA ? "fasta" : "arrow");
        }
      const uint8_t *slash = (const uint8_t *) memchr(head.data(),'/',(size_t) (nl - head.data()));
      if (slash == NULL) return dx_fail(ctx,DX_E_FORMAT,"Header line incorrectly formatted ?");
      plen = (int32_t) (slash - head.data());
      hbytes = 2 + 4 + (size_t) plen;
    }
  else if (head[0] != '>')
    return dx_fail(ctx,DX_E_ARG,"dx_dexta_part_dev: a part without the file header must start at an entry header ('>')");

  int64_t *d_hdr = NULL, nent = 0;
  if ((rc = dxk_index_positions(ctx,DX_PRED_FASTA_HDR,d_text,n,0,&d_hdr,&nent)) != DX_OK) return rc;

  FaEntries ent;
  ent.n = nent;
  const size_t N = (size_t) nent;
  ent.hdr    = (int64_t *) dx_arena_get(ctx,N*8);
  ent.seq    = (int64_t *) dx_arena_get(ctx,N*8);
  ent.region = (int64_t *) dx_arena_get(ctx,N*8);
  ent.off    = (int64_t *) dx_arena_get(ctx,(N+1)*8);
  ent.rlen   = (int32_t *) dx_arena_get(ctx,N*4);
  ent.width  = (int32_t *) dx_arena_get(ctx,N*4);
  ent.well   = (int32_t *) dx_arena_get(ctx,N*4);
  ent.beg    = (int32_t *) dx_arena_get(ctx,N*4);
  ent.end    = (int32_t *) dx_arena_get(ctx,N*4);
  ent.aux    = (int32_t *) dx_arena_get(ctx,N*8);
  ent.flag   = (int32_t *) dx_arena_get(ctx,N*4);
  ent.bytes  = (uint32_t *) dx_arena_get(ctx,N*4);
  if (!ent.hdr || !ent.seq || !ent.region || !ent.off || !ent.rlen || !ent.width || !ent.well ||
      !ent.beg || !ent.end || !ent.aux || !ent.flag || !ent.bytes) return DX_E_NOMEM;

  int32_t *d_flags = (int32_t *) dx_arena_get(ctx,32);            // [0] any flag, [1] pack error, [2..3] ticket
  if (d_flags == NULL) return DX_E_NOMEM;
  DX_CUDA(ctx,cudaMemsetAsync(d_flags,0,32,ctx->stream));
  int32_t anyflag = 1;
  if (exact)
    { if ((rc = dxk_fa_measure(ctx,kind,d_text,n,d_hdr,ent)) != DX_OK) return rc; }
  else
    { if ((rc = dxk_fa_measure2(ctx,kind,d_text,n,d_hdr,ent,d_flags)) != DX_OK) return rc;
      DX_CUDA(ctx,cudaMemcpyAsync(&anyflag,d_flags,4,cudaMemcpyDeviceToHost,ctx->stream));
      DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
    }

  // entries the device could not settle: non-canonical headers go through the host's sscanf
  std::vector<int32_t> flag;
  if (anyflag)
    { if ((rc = download(ctx,ent.flag,N,flag)) != DX_OK) return rc; }
  else
    flag.assign(N,0);
  for (size_t e = 0; e < N && anyflag; e++)
    { if (flag[e] & 4)
        return dx_fail(ctx,DX_E_TOOLONG,"%s line is too long (> 99998 chars) or unterminated (entry %lld)",
                       kind == DX_FASTA ? "Fasta" : "Arrow",(long long) (ctx->origin_entry + (int64_t) e + 1));
      if (!(flag[e] & 1)) continue;
      int64_t h0 = 0;
      DX_CUDA(ctx,cudaMemcpyAsync(&h0,ent.hdr+e,8,cudaMemcpyDeviceToHost,ctx->stream));
      DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
      std::vector<uint8_t> line;
      if ((rc = peek(ctx,d_text,n,(size_t) h0,100000,line)) != DX_OK) return rc;
      const uint8_t *e1 = (const uint8_t *) memchr(line.data(),'\n',line.size());
      if (e1 == NULL)
        return dx_fail(ctx,DX_E_TOOLONG,"header line too long (entry %lld)",(long long) (ctx->origin_entry + (int64_t) e + 1));
      std::vector<char> txt(line.begin(),line.begin() + (e1 - line.data()) + 1);
      txt.push_back('\0');
      char *sl = strchr(txt.data()+1,'/');
      if (sl == NULL) return dx_fail(ctx,DX_E_FORMAT,"Header line incorrectly formatted ?");
      int32_t well = 0, beg = 0, en = 0, aux[2] = { 0, 0 };
      if (kind == DX_FASTA)
        { int qv = 0;
          int x = sscanf(sl+1,"%d/%d_%d RQ=0.%d\n",&well,&beg,&en,&qv);      // dexta.c:151
          if (x < 3) return dx_fail(ctx,DX_E_FORMAT,"Header line incorrectly formatted ?");
          aux[0] = (x == 3) ? 0 : qv;
        }
      else
        { float snr[4];
          int x = sscanf(sl+1,"%d/%d_%d SN=%f,%f,%f,%f\n",&well,&beg,&en,snr,snr+1,snr+2,snr+3);
          if (x != 7) return dx_fail(ctx,DX_E_FORMAT,"Header line incorrectly formatted ?");
          uint32_t c[4];
          for (int k = 0; k < 4; k++)                                           // dexar.c:159-163
            c[k] = (snr[k] > 99.99) ? 9999u : ((uint32_t) (snr[k]*100.) & 0xffffu);
          aux[0] = (int32_t) (c[0] | (c[1] << 16));
          aux[1] = (int32_t) (c[2] | (c[3] << 16));
        }
      if ((rc = upload(ctx,ent.well+e,&well,1)) != DX_OK) return rc;
      if ((rc = upload(ctx,ent.beg+e,&beg,1)) != DX_OK) return rc;
      if ((rc = upload(ctx,ent.end+e,&en,1)) != DX_OK) return rc;
      if ((rc = upload(ctx,ent.aux+2*e,aux,2)) != DX_OK) return rc;
    }

  int64_t body = 0;
  if ((rc = dxk_fa_offsets(ctx,kind,ent,lwell_in,&body)) != DX_OK) return rc;
  if (hbytes + (size_t) body > cap)
    return dx_fail_cap(ctx,(size_t) (hbytes + (size_t) body),cap);

  if (with_header)
    { std::vector<uint8_t> fh(hbytes);
      const uint16_t key = 0x55aa;
      memcpy(fh.data(),&key,2);
      memcpy(fh.data()+2,&plen,4);
      memcpy(fh.data()+6,head.data(),(size_t) plen);
      if ((rc = upload(ctx,d_out,fh.data(),hbytes)) != DX_OK) return rc;
    }
  if (exact)
    { if ((rc = dxk_fa_pack(ctx,kind,d_text,n,ent,lwell_in,d_out + hbytes)) != DX_OK) return rc;
      DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
    }
  else
    { // d_flags: [1] pack error, [2..3] ticket, [4] entries left to k_fa_pack2, [6..7] its ticket
      int32_t res[4] = { 0, 0, 0, 0 };
      if (ctx->route[DXR_PACK2])
        rc = dxk_fa_pack2(ctx,kind,d_text,ent,lwell_in,d_out + hbytes,d_flags + 1,(unsigned long long *) (d_flags + 2),0);
      else
        rc = dxk_fa_pack3(ctx,kind,d_text,n,ent,lwell_in,d_out + hbytes,d_flags + 1,d_flags + 4,
                          (unsigned long long *) (d_flags + 2));
      if (rc != DX_OK) return rc;
      DX_CUDA(ctx,cudaMemcpyAsync(res,d_flags + 1,16,cudaMemcpyDeviceToHost,ctx->stream));
      DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
      if (res[0] == 2) return dx_fail(ctx,DX_E_TOOLONG,"%s line is too long (> 99998 chars)",kind == DX_FASTA ? "Fasta" : "Arrow");
      if (res[0]) { *redo = true; return DX_OK; }
      if (res[3])                                   // entries off the lattice (or narrower than 16)
        { if ((rc = dxk_fa_pack2(ctx,kind,d_text,ent,lwell_in,d_out + hbytes,d_flags + 1,
                                 (unsigned long long *) (d_flags + 6),1)) != DX_OK) return rc;
          DX_CUDA(ctx,cudaMemcpyAsync(res,d_flags + 1,4,cudaMemcpyDeviceToHost,ctx->stream));
          DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
          if (res[0] == 2) return dx_fail(ctx,DX_E_TOOLONG,"%s line is too long (> 99998 chars)",kind == DX_FASTA ? "Fasta" : "Arrow");
          if (res[0]) { *redo = true; return DX_OK; }
        }
    }
  if (last_well != NULL)
    { *last_well = lwell_in;
      if (N > 0)
        { DX_CUDA(ctx,cudaMemcpyAsync(last_well,ent.well + (N - 1),4,cudaMemcpyDeviceToHost,ctx->stream));
          DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
        }
    }
  ctx->last_entries = nent;
  *out_len = hbytes + (size_t) body;
  return DX_OK;
}

// Everything undexta needs to know about a 2-bit image before the payload is touched.
struct PkPlan
{ std::vector<PkDecEntry> ent;
  std::vector<char>       prefix;
  size_t                  text_len;
};

static int plan_undexta(dx_ctx *ctx, int kind, const uint8_t *d_in, size_t n, int width, PkPlan &plan)
{ int rc;
  if (width <= 0) return dx_fail(ctx,DX_E_ARG,"line width must be positive");
  std::vector<uint8_t> head;
  if ((rc = peek(ctx,d_in,n,0,6,head)) != DX_OK) return rc;
  if (head.size() < 6) return dx_fail(ctx,DX_E_TRUNC,"System error, read failed!");
  uint16_t key; memcpy(&key,head.data(),2);
  int32_t  plen; memcpy(&plen,head.data()+2,4);
  const bool legacy = (kind == DX_FASTA && (key == 0x33cc || key == 0xcc33));
  const bool flip   = (key == 0xaa55 || key == 0xcc33);
  if (!(key == 0x55aa || key == 0xaa55 || legacy))
    return dx_fail(ctx,DX_E_KEY,"Not a %s file, endian key invalid",kind == DX_FASTA ? ".dexta" : ".dexar");
  if (flip) plen = (int32_t) __builtin_bswap32((uint32_t) plen);
  if (plen < 0 || (size_t) plen + 6 > n) return dx_fail(ctx,DX_E_TRUNC,"System error, read failed!");
  if ((rc = peek(ctx,d_in,n,6,(size_t) plen,head)) != DX_OK) return rc;
  plan.prefix.assign(head.begin(),head.end());
  const size_t first = 6 + (size_t) plen;
  const int fieldbytes = (kind == DX_FASTA) ? 12 : 16;

  struct Hdr { int64_t q; int32_t well, beg, end, aux[2]; };
  std::vector<Hdr> hdrs;

  if (legacy || flip)
    { // old 16-bit layout or foreign byte order (undexta.c:140-155, 211-240): rare, so the
      // header chain is hopped on the host over a copy of the image
      std::vector<uint8_t> img;
      if ((rc = peek(ctx,d_in,n,0,n,img)) != DX_OK) return rc;
      size_t at = first;
      int32_t well = 0;
      while (at < n)
        { uint8_t b = img[at++];
          while (b == 255)
            { well += 255;
              if (at >= n) return dx_fail(ctx,DX_E_TRUNC,"System error, read failed!");
              b = img[at++];
            }
          well += b;
          Hdr h; h.well = well; h.aux[0] = h.aux[1] = 0;
          if (legacy)
            { if (at + 6 > n) return dx_fail(ctx,DX_E_TRUNC,"System error, read failed!");
              uint16_t v[3]; memcpy(v,img.data()+at,6);
              if (flip) for (int k = 0; k < 3; k++) v[k] = (uint16_t) ((v[k] >> 8) | (v[k] << 8));
              h.beg = v[0]; h.end = v[1]; h.aux[0] = v[2];
              at += 6;
            }
          else
            { if (at + (size_t) fieldbytes > n) return dx_fail(ctx,DX_E_TRUNC,"System error, read failed!");
              uint32_t v[2]; memcpy(v,img.data()+at,8);
              h.beg = (int32_t) __builtin_bswap32(v[0]); h.end = (int32_t) __builtin_bswap32(v[1]);
              if (kind == DX_FASTA)
                { uint32_t qv; memcpy(&qv,img.data()+at+8,4); h.aux[0] = (int32_t) __builtin_bswap32(qv); }
              else
                { uint16_t c[4]; memcpy(c,img.data()+at+8,8);
                  for (int k = 0; k < 4; k++) c[k] = (uint16_t) ((c[k] >> 8) | (c[k] << 8));
                  h.aux[0] = (int32_t) (c[0] | ((uint32_t) c[1] << 16));
                  h.aux[1] = (int32_t) (c[2] | ((uint32_t) c[3] << 16));
                }
              at += (size_t) fieldbytes;
            }
          h.q = (int64_t) at;                         // here: first payload byte
          const int64_t rlen = (int64_t) h.end - h.beg;
          if (rlen < 0) return dx_fail(ctx,DX_E_FORMAT,"negative read length in entry header");
          at += (size_t) ((rlen + 3) >> 2);
          if (at > n) return dx_fail(ctx,DX_E_TRUNC,"System error, read failed!");
          hdrs.push_back(h);
        }
    }
  else
    { int64_t *d_q = NULL, nc = 0;
      if ((rc = dxk_index_positions(ctx,kind == DX_FASTA ? DX_PRED_QVCAND : DX_PRED_ARCAND,
                                    d_in,n,first + 1,&d_q,&nc)) != DX_OK) return rc;
      int64_t  *d_end  = (int64_t *) dx_arena_get(ctx,(size_t) nc*8);
      CandInfo *d_info = (CandInfo *) dx_arena_get(ctx,(size_t) nc*sizeof(CandInfo));
      if (!d_end || !d_info) return DX_E_NOMEM;
      if ((rc = dxk_pk_walk(ctx,fieldbytes,d_in,n,d_q,nc,d_end)) != DX_OK) return rc;
      if ((rc = dxk_cand_context(ctx,d_in,n,first,d_q,nc,fieldbytes,d_info)) != DX_OK) return rc;
      std::vector<int64_t> q, end;
      std::vector<CandInfo> info;
      if ((rc = download(ctx,d_q,(size_t) nc,q)) != DX_OK) return rc;
      if ((rc = download(ctx,d_end,(size_t) nc,end)) != DX_OK) return rc;
      if ((rc = download(ctx,d_info,(size_t) nc,info)) != DX_OK) return rc;
      PkWalkUser user = { fieldbytes, d_in, n };
      std::vector<ChainEntry> chain;
      if ((rc = resolve_chain(ctx,d_in,n,first,fieldbytes,q,end,info,pk_walk_one,&user,chain)) != DX_OK)
        return rc;
      hdrs.reserve(chain.size());
      for (const ChainEntry &c : chain)
        { Hdr h; h.well = c.well;
          h.beg = le32(c.field); h.end = le32(c.field+4);
          h.aux[0] = le32(c.field+8);
          h.aux[1] = (kind == DX_ARROW) ? le32(c.field+12) : 0;
          h.q = c.q + fieldbytes;
          hdrs.push_back(h);
        }
    }

  // output layout: "%s/%d/%d_%d RQ=0.%d\n" + wrapped sequence (undexta.c:242-270)
  size_t at = 0;
  plan.ent.resize(hdrs.size());
  for (size_t i = 0; i < hdrs.size(); i++)
    { const Hdr &h = hdrs[i];
      PkDecEntry &d = plan.ent[i];
      d.bin_off = h.q; d.out_off = (int64_t) at;
      d.well = h.well; d.beg = h.beg; d.end = h.end; d.aux[0] = h.aux[0]; d.aux[1] = h.aux[1];
      size_t hl = plan.prefix.size() + 1 + ndigits(h.well) + 1 + ndigits(h.beg) + 1 + ndigits(h.end);
      if (kind == DX_FASTA)
        hl += 6 + ndigits(h.aux[0]) + 1;
      else
        { hl += 4;
          for (int k = 0; k < 4; k++)
            { const uint32_t c = ((uint32_t) h.aux[k >> 1] >> (16*(k & 1))) & 0xffffu;
              hl += ndigits((int32_t) (c / 100)) + 3 + (k < 3);
            }
          hl += 1;
        }
      at += hl;
      d.text_off = (int64_t) at;
      const int64_t rlen = (int64_t) h.end - h.beg;
      if (rlen > 0)
        at += (size_t) (rlen + (rlen + width - 1) / width);
    }
  plan.text_len = at;
  return DX_OK;
}

// The usual case of dx_undexta_dev (current key, native byte order, width >= 16) with everything but
// the verification of the entry chain on the device.  *handled = false: take the general path.
// d_out == NULL: only the size of the text is wanted.
static int undexta_fast(dx_ctx *ctx, int kind, const uint8_t *d_in, size_t n, int width, int upper,
                        uint8_t *d_out, size_t cap, size_t *out_len, bool *handled)
{ int rc;
  *handled = false;
  if (width < 16 || ctx->route[DXR_NO_FAST]) return DX_OK;
  std::vector<uint8_t> head;
  if ((rc = peek(ctx,d_in,n,0,6,head)) != DX_OK) return rc;
  if (head.size() < 6) return DX_OK;
  uint16_t key; memcpy(&key,head.data(),2);
  int32_t  plen; memcpy(&plen,head.data()+2,4);
  if (key != 0x55aa || plen < 0 || (size_t) plen + 6 > n) return DX_OK;
  const size_t first = 6 + (size_t) plen;
  const int fieldbytes = (kind == DX_FASTA) ? 12 : 16;
  char *d_prefix = (char *) dx_arena_get(ctx,(size_t) plen + 1);
  if (d_prefix == NULL) return DX_E_NOMEM;
  DX_CUDA(ctx,cudaMemcpyAsync(d_prefix,d_in + 6,(size_t) plen,cudaMemcpyDeviceToDevice,ctx->stream));

  int64_t *d_q = NULL, nc = 0;
  if ((rc = dxk_index_positions(ctx,kind == DX_FASTA ? DX_PRED_QVCAND : DX_PRED_ARCAND,
                                d_in,n,first + 1,&d_q,&nc)) != DX_OK) return rc;
  const size_t N = (size_t) nc;
  if (N == 0) return DX_OK;
  int64_t *d_end   = (int64_t *) dx_arena_get(ctx,N*8);
  int32_t *d_ffrun = (int32_t *) dx_arena_get(ctx,N*4);
  uint8_t *d_last  = (uint8_t *) dx_arena_get(ctx,N);
  if (!d_end || !d_ffrun || !d_last) return DX_E_NOMEM;
  if ((rc = dxk_pk_cand_prep(ctx,d_in,n,first,fieldbytes,d_q,nc,d_end,d_ffrun,d_last)) != DX_OK) return rc;
  int64_t *h_q     = (int64_t *) dx_hpin_get(ctx,N*8);
  int64_t *h_end   = (int64_t *) dx_hpin_get(ctx,N*8);
  int32_t *h_ffrun = (int32_t *) dx_hpin_get(ctx,N*4);
  uint8_t *h_last  = (uint8_t *) dx_hpin_get(ctx,N);
  int32_t *h_cand  = (int32_t *) dx_hpin_get(ctx,N*4);
  int32_t *h_well  = (int32_t *) dx_hpin_get(ctx,N*4);
  int64_t *h_total = (int64_t *) dx_hpin_get(ctx,8);
  if (!h_q || !h_end || !h_ffrun || !h_last || !h_cand || !h_well || !h_total) return DX_E_NOMEM;
  DX_CUDA(ctx,cudaMemcpyAsync(h_q,d_q,N*8,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaMemcpyAsync(h_end,d_end,N*8,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaMemcpyAsync(h_ffrun,d_ffrun,N*4,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaMemcpyAsync(h_last,d_last,N,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));

  size_t M = 0;                                          // the chain (see resolve_chain)
  { int64_t cur = (int64_t) first;
    int32_t well = 0;
    size_t i = 0;
    while (cur < (int64_t) n)
      { while (i < N && h_q[i] - 1 < cur) i++;
        while (i < N && h_last[i] == 0xff && h_q[i] - 1 - cur <= h_ffrun[i]) i++;
        if (i >= N || h_end[i] < 0) return DX_OK;
        const int64_t gap = h_q[i] - 1 - cur;
        if (gap > h_ffrun[i] || h_last[i] == 0xff) return DX_OK;
        if (h_end[i] > (int64_t) n || h_end[i] <= cur) return DX_OK;
        well += 255 * (int32_t) gap + h_last[i];
        h_cand[M] = (int32_t) i; h_well[M] = well; M++;
        cur = h_end[i];
        i++;
      }
  }
  int32_t *d_cand = (int32_t *) dx_arena_get(ctx,M*4 + 4);
  int32_t *d_well = (int32_t *) dx_arena_get(ctx,M*4 + 4);
  uint32_t *d_len = (uint32_t *) dx_arena_get(ctx,M*4 + 4);
  int64_t *d_opre = (int64_t *) dx_arena_get(ctx,(M+1)*8);
  PkDecEntry *d_ent = (PkDecEntry *) dx_arena_get(ctx,(M+1)*sizeof(PkDecEntry));
  unsigned long long *d_ticket = (unsigned long long *) dx_arena_get(ctx,8);
  if (!d_cand || !d_well || !d_len || !d_opre || !d_ent || !d_ticket) return DX_E_NOMEM;
  DX_CUDA(ctx,cudaMemsetAsync(d_ticket,0,8,ctx->stream));
  if (M > 0)
    { DX_CUDA(ctx,cudaMemcpyAsync(d_cand,h_cand,M*4,cudaMemcpyHostToDevice,ctx->stream));
      DX_CUDA(ctx,cudaMemcpyAsync(d_well,h_well,M*4,cudaMemcpyHostToDevice,ctx->stream));
    }
  if ((rc = dxk_pk_layout(ctx,kind,d_in,d_q,d_cand,d_well,(int64_t) M,fieldbytes,plen,width,d_len,d_opre,d_ent)) != DX_OK)
    return rc;
  DX_CUDA(ctx,cudaMemcpyAsync(h_total,d_opre+M,8,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  const size_t total = (size_t) *h_total;
  if (d_out != NULL)
    { if (total > cap) return dx_fail_cap(ctx,(size_t) (total),cap);
      if (ctx->route[DXR_PACK2])
        rc = dxk_unpack2(ctx,kind,upper,width,d_in,n,d_ent,(int64_t) M,d_prefix,plen,d_out,d_ticket);
      else
        rc = dxk_unpack3(ctx,kind,upper,width,d_in,n,d_ent,(int64_t) M,d_prefix,plen,d_out,d_ticket);
      if (rc != DX_OK) return rc;
      DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
    }
  *out_len = total;
  *handled = true;
  return DX_OK;
}

extern "C" int dx_undexta_dev(dx_ctx *ctx, int kind, const uint8_t *d_in, size_t n, int width,
                              int upper, uint8_t *d_out, size_t cap, size_t *out_len)
{ if (ctx == NULL || out_len == NULL || (kind != DX_FASTA && kind != DX_ARROW)) return DX_E_ARG;
  *out_len = 0;
  int rc;
  if ((rc = check_buf(ctx,d_in,"image")) != DX_OK) return rc;
  cudaSetDevice(ctx->device);
  dx_arena_reset(ctx);
  { bool handled = false;
    if (d_out != NULL && (rc = undexta_fast(ctx,kind,d_in,n,width,upper,d_out,cap,out_len,&handled)) != DX_OK)
      return rc;
    if (handled) return DX_OK;
    dx_arena_reset(ctx);
  }
  PkPlan plan;
  if ((rc = plan_undexta(ctx,kind,d_in,n,width,plan)) != DX_OK) return rc;
  if (plan.text_len > cap)
    return dx_fail_cap(ctx,(size_t) (plan.text_len),cap);
  if (d_out == NULL && plan.text_len > 0) return dx_fail(ctx,DX_E_ARG,"output is NULL");
  const size_t N = plan.ent.size();
  PkDecEntry *d_ent = (PkDecEntry *) dx_arena_get(ctx,N*sizeof(PkDecEntry));
  char *d_prefix = (char *) dx_arena_get(ctx,plan.prefix.size()+1);
  if (!d_ent || !d_prefix) return DX_E_NOMEM;
  if ((rc = upload(ctx,d_ent,plan.ent.data(),N)) != DX_OK) return rc;
  if ((rc = upload(ctx,d_prefix,plan.prefix.data(),plan.prefix.size())) != DX_OK) return rc;
  if ((rc = dxk_unpack(ctx,kind,upper,width,d_in,d_ent,(int64_t) N,d_prefix,(int) plan.prefix.size(),
                       d_out)) != DX_OK) return rc;
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  *out_len = plan.text_len;
  return DX_OK;
}

extern "C" int dx_undexta_size_dev(dx_ctx *ctx, int kind, const uint8_t *d_in, size_t n, int width,
                                   size_t *out_len)
{ if (ctx == NULL || out_len == NULL || (kind != DX_FASTA && kind != DX_ARROW)) return DX_E_ARG;
  *out_len = 0;
  int rc;
  if ((rc = check_buf(ctx,d_in,"image")) != DX_OK) return rc;
  cudaSetDevice(ctx->device);
  dx_arena_reset(ctx);
  { bool handled = false;
    if ((rc = undexta_fast(ctx,kind,d_in,n,width,0,NULL,0,out_len,&handled)) != DX_OK) return rc;
    if (handled) return DX_OK;
    dx_arena_reset(ctx);
  }
  PkPlan plan;
  if ((rc = plan_undexta(ctx,kind,d_in,n,width,plan)) != DX_OK) return rc;
  *out_len = plan.text_len;
  return DX_OK;
}

// ---- one window of a .dexta / .dexar image ----------------------------------------------------------
// The chain is walked from a carried position and well (dx_chain_walk_general); an entry the candidates
// do not give is read by itself, and the walk ends in front of the first entry that does not lie wholly
// in the buffer.

struct PkWinSlow { dx_ctx *ctx; const uint8_t *d_buf; size_t n; int fieldbytes; int64_t need; };

// the entry at buffer offset cur read by itself; DX_E_CAP (u.need: the buffer offset it needs) when its
// delta bytes, fields or payload reach past the buffer
static int pk_win_slow(void *user, int64_t cur, int64_t *q, int64_t *end, int32_t *delta)
{ PkWinSlow &u = *(PkWinSlow *) user;
  std::vector<uint8_t> win;
  int64_t p = cur;
  int32_t add = 0;
  int rc;
  for (;;)
    { if ((rc = peek(u.ctx,u.d_buf,u.n,(size_t) p,4096,win)) != DX_OK) return rc;
      size_t k = 0;
      while (k < win.size() && win[k] == 0xff) k++;
      add += 255 * (int32_t) k; p += (int64_t) k;
      if (k < win.size()) { add += win[k]; p += 1; break; }
      if (p >= (int64_t) u.n)                               // a delta is at most 2^31 wells: 8 421 505 bytes
        { u.need = cur + 8421505 + u.fieldbytes; return DX_E_CAP; }
    }
  if ((rc = peek(u.ctx,u.d_buf,u.n,(size_t) p,(size_t) u.fieldbytes,win)) != DX_OK) return rc;
  if ((int) win.size() < u.fieldbytes) { u.need = p + u.fieldbytes; return DX_E_CAP; }
  const int64_t rlen = (int64_t) le32(win.data()+4) - le32(win.data());
  if (rlen < 0) return dx_fail(u.ctx,DX_E_FORMAT,"negative read length in entry header");
  *q = p; *end = p + u.fieldbytes + ((rlen + 3) >> 2); *delta = add;
  if (*end > (int64_t) u.n) { u.need = *end; return DX_E_CAP; }
  return DX_OK;
}

extern "C" int dx_undexta_window_dev(dx_ctx *ctx, int kind, const uint8_t *h_head, size_t head_n,
                                     const uint8_t *d_buf, size_t buf_n, int64_t buf_off, int64_t cur_in,
                                     int32_t well_in, int is_last, int width, int upper, uint8_t *d_out, size_t cap,
                                     size_t *out_len, int64_t *cur_out, int32_t *well_out)
{ if (ctx == NULL || out_len == NULL || cur_out == NULL || well_out == NULL || (kind != DX_FASTA && kind != DX_ARROW))
    return DX_E_ARG;
  *out_len = 0; *cur_out = cur_in; *well_out = well_in;
  ctx->last_entries = 0;
  int rc;
  if (h_head == NULL) return dx_fail(ctx,DX_E_ARG,"dx_undexta_window_dev: h_head is NULL");
  if (width <= 0) return dx_fail(ctx,DX_E_ARG,"line width must be positive");
  if (head_n < 6) return dx_fail(ctx,DX_E_TRUNC,"System error, read failed!");
  uint16_t key; memcpy(&key,h_head,2);
  int32_t  plen; memcpy(&plen,h_head+2,4);
  if (!(key == 0x55aa || key == 0xaa55 || (kind == DX_FASTA && (key == 0x33cc || key == 0xcc33))))
    return dx_fail(ctx,DX_E_KEY,"Not a %s file, endian key invalid",kind == DX_FASTA ? ".dexta" : ".dexar");
  if (key != 0x55aa)
    return dx_fail(ctx,DX_E_FORMAT,"%s image: windows take images of the 0x55aa layout in the native byte order; "
                   "decode it whole with dx_undexta_dev",key == 0xaa55 ? "a foreign-endian" : "an old-layout (0x33cc)");
  if (plen < 0 || (size_t) plen + 6 > head_n) return dx_fail(ctx,DX_E_TRUNC,"System error, read failed!");
  if ((rc = check_buf(ctx,d_buf,"window buffer")) != DX_OK) return rc;
  const int64_t first = 6 + (int64_t) plen, buf_end = buf_off + (int64_t) buf_n;
  if (buf_off < 0 || cur_in < first || cur_in < buf_off || cur_in > buf_end)
    return dx_fail(ctx,DX_E_ARG,"dx_undexta_window_dev: the chain position %lld is not in the buffer [%lld, %lld) "
                   "behind the header (%lld bytes)",(long long) cur_in,(long long) buf_off,(long long) buf_end,(long long) first);
  cudaSetDevice(ctx->device);
  dx_arena_reset(ctx);
  const int fieldbytes = (kind == DX_FASTA) ? 12 : 16;
  const int64_t s = cur_in - buf_off;

  int64_t *d_q = NULL, nc = 0;
  if (s < (int64_t) buf_n &&
      (rc = dxk_index_positions(ctx,kind == DX_FASTA ? DX_PRED_QVCAND : DX_PRED_ARCAND,d_buf,buf_n,(size_t) s + 1,
                                &d_q,&nc)) != DX_OK) return rc;
  const size_t N = (size_t) nc;
  int64_t *d_end   = (int64_t *) dx_arena_get(ctx,N*8);
  int32_t *d_ffrun = (int32_t *) dx_arena_get(ctx,N*4);
  uint8_t *d_last  = (uint8_t *) dx_arena_get(ctx,N);
  int64_t *h_q     = (int64_t *) dx_hpin_get(ctx,N*8);
  int64_t *h_end   = (int64_t *) dx_hpin_get(ctx,N*8);
  int32_t *h_ffrun = (int32_t *) dx_hpin_get(ctx,N*4);
  uint8_t *h_last  = (uint8_t *) dx_hpin_get(ctx,N);
  if (!d_end || !d_ffrun || !d_last || !h_q || !h_end || !h_ffrun || !h_last) return DX_E_NOMEM;
  if (N > 0)
    { if ((rc = dxk_pk_cand_prep(ctx,d_buf,buf_n,(size_t) s,fieldbytes,d_q,nc,d_end,d_ffrun,d_last)) != DX_OK) return rc;
      DX_CUDA(ctx,cudaMemcpyAsync(h_q,d_q,N*8,cudaMemcpyDeviceToHost,ctx->stream));
      DX_CUDA(ctx,cudaMemcpyAsync(h_end,d_end,N*8,cudaMemcpyDeviceToHost,ctx->stream));
      DX_CUDA(ctx,cudaMemcpyAsync(h_ffrun,d_ffrun,N*4,cudaMemcpyDeviceToHost,ctx->stream));
      DX_CUDA(ctx,cudaMemcpyAsync(h_last,d_last,N,cudaMemcpyDeviceToHost,ctx->stream));
      DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
    }
  std::vector<int32_t> stat(N);                         // the walk's view of a candidate: did it end in the buffer
  std::vector<int64_t> soff(6*N);
  for (size_t i = 0; i < N; i++) { stat[i] = (h_end[i] < 0); soff[6*i + 5] = h_end[i]; }
  const DxChainIn ci = { h_q, h_ffrun, h_last, stat.data(), soff.data(), NULL, (int64_t) N, s, (int64_t) buf_n,
                         s, (int64_t) buf_n };
  PkWinSlow u = { ctx, d_buf, buf_n, fieldbytes, 0 };
  std::vector<DxChainEntry> ent;
  int64_t stop = s;
  rc = dx_chain_walk_general(ci,well_in,pk_win_slow,&u,ent,&stop);
  if (rc == DX_E_CAP)                                   // the walk stopped in front of an entry the buffer cuts
    { if (is_last) return dx_fail(ctx,DX_E_TRUNC,"System error, read failed!");
      if (ent.empty())
        { dx_fail(ctx,DX_E_CAP,"the entry at image offset %lld runs past the end of the buffer (%lld): it needs the image "
                  "up to %lld",(long long) cur_in,(long long) buf_end,(long long) (buf_off + u.need));
          ctx->need_bytes = (size_t) (buf_off + u.need);
          return DX_E_CAP;
        }
      stop = ent.back().end;
    }
  else if (rc != DX_OK)
    return rc;

  const size_t M = ent.size();
  *cur_out = buf_off + stop;
  *well_out = (M > 0) ? ent.back().well : well_in;
  ctx->last_entries = (int64_t) M;
  if (M == 0) return DX_OK;
  int64_t *h_qm  = (int64_t *) dx_hpin_get(ctx,M*8);
  int32_t *h_cw  = (int32_t *) dx_hpin_get(ctx,M*8);     // [0, M) candidate = m, [M, 2M) well
  int64_t *h_total = (int64_t *) dx_hpin_get(ctx,8);
  int64_t *d_qm  = (int64_t *) dx_arena_get(ctx,M*8);
  int32_t *d_cw  = (int32_t *) dx_arena_get(ctx,M*8);
  uint32_t *d_len = (uint32_t *) dx_arena_get(ctx,M*4);
  int64_t *d_opre = (int64_t *) dx_arena_get(ctx,(M+1)*8);
  PkDecEntry *d_ent = (PkDecEntry *) dx_arena_get(ctx,(M+1)*sizeof(PkDecEntry));
  char *d_prefix = (char *) dx_arena_get(ctx,(size_t) plen + 1);
  unsigned long long *d_ticket = (unsigned long long *) dx_arena_get(ctx,8);
  if (!h_qm || !h_cw || !h_total || !d_qm || !d_cw || !d_len || !d_opre || !d_ent || !d_prefix || !d_ticket)
    return DX_E_NOMEM;
  for (size_t m = 0; m < M; m++) { h_qm[m] = ent[m].q; h_cw[m] = (int32_t) m; h_cw[M + m] = ent[m].well; }
  DX_CUDA(ctx,cudaMemcpyAsync(d_qm,h_qm,M*8,cudaMemcpyHostToDevice,ctx->stream));
  DX_CUDA(ctx,cudaMemcpyAsync(d_cw,h_cw,M*8,cudaMemcpyHostToDevice,ctx->stream));
  if (plen > 0) DX_CUDA(ctx,cudaMemcpyAsync(d_prefix,h_head + 6,(size_t) plen,cudaMemcpyHostToDevice,ctx->stream));
  DX_CUDA(ctx,cudaMemsetAsync(d_ticket,0,8,ctx->stream));
  if ((rc = dxk_pk_layout(ctx,kind,d_buf,d_qm,d_cw,d_cw + M,(int64_t) M,fieldbytes,plen,width,d_len,d_opre,d_ent)) != DX_OK)
    return rc;
  DX_CUDA(ctx,cudaMemcpyAsync(h_total,d_opre + M,8,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  const size_t total = (size_t) *h_total;
  if (total > cap) return dx_fail_cap(ctx,total,cap);
  if (d_out == NULL) return dx_fail(ctx,DX_E_ARG,"output is NULL");
  if (width < 16)
    rc = dxk_unpack(ctx,kind,upper,width,d_buf,d_ent,(int64_t) M,d_prefix,plen,d_out);
  else if (ctx->route[DXR_PACK2])
    rc = dxk_unpack2(ctx,kind,upper,width,d_buf,buf_n,d_ent,(int64_t) M,d_prefix,plen,d_out,d_ticket);
  else
    rc = dxk_unpack3(ctx,kind,upper,width,d_buf,buf_n,d_ent,(int64_t) M,d_prefix,plen,d_out,d_ticket);
  if (rc != DX_OK) return rc;
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  *out_len = total;
  return DX_OK;
}

extern "C" int dx_compress_reads_dev(dx_ctx *ctx, int kind, const uint8_t *d_src,
                                     const int64_t *d_src_off, const int32_t *d_len, int64_t nreads,
                                     uint8_t *d_dst, const int64_t *d_dst_off)
{ if (ctx == NULL || nreads < 0) return DX_E_ARG;
  cudaSetDevice(ctx->device);
  dx_arena_reset(ctx);
  if (ctx->route[DXR_EXACT_PACK])
    return dxk_compress_reads(ctx,kind,d_src,d_src_off,d_len,nreads,d_dst,d_dst_off);
  return dxk_compress_reads2(ctx,kind,d_src,d_src_off,d_len,nreads,d_dst,d_dst_off);
}

extern "C" int dx_uncompress_reads_dev(dx_ctx *ctx, int kind, int upper, const uint8_t *d_src,
                                       const int64_t *d_src_off, const int32_t *d_len,
                                       int64_t nreads, uint8_t *d_dst, const int64_t *d_dst_off)
{ if (ctx == NULL || nreads < 0) return DX_E_ARG;
  cudaSetDevice(ctx->device);
  dx_arena_reset(ctx);
  if (ctx->route[DXR_EXACT_PACK])
    return dxk_uncompress_reads(ctx,kind,upper,d_src,d_src_off,d_len,nreads,d_dst,d_dst_off);
  return dxk_uncompress_reads2(ctx,kind,upper,d_src,d_src_off,d_len,nreads,d_dst,d_dst_off);
}

// ================================================================================================
//  QV coder: scan
// ================================================================================================

static int qv_frame(dx_ctx *ctx, const uint8_t *d_text, size_t n, uint64_t *totchar)
{ int rc;
  ctx->qv_text = NULL; ctx->qv_n = 0; ctx->qv_ent.n = 0;
  *totchar = 0;
  if (n == 0) { ctx->qv_text = d_text; return DX_OK; }

  int64_t *d_nl = NULL, nlines = 0;
  if ((rc = dxk_index_positions(ctx,DX_PRED_NEWLINE,d_text,n,0,&d_nl,&nlines)) != DX_OK) return rc;
  // the text must end with a newline; in the usual case (complete entries) k_qv_entries reports the
  // last newline together with its other results, so there is no extra round trip for it
  if (nlines % 6 != 0 || nlines == 0)
    { int64_t last = -1;
      if (nlines > 0)
        { DX_CUDA(ctx,cudaMemcpyAsync(&last,d_nl+nlines-1,8,cudaMemcpyDeviceToHost,ctx->stream));
          DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
        }
      ctx->err_line = ctx->origin_line + nlines + 1;
      if (last != (int64_t) n - 1)
        return dx_fail(ctx,DX_E_FORMAT,"Line %lld: Last line does not end with a newline !",
                       (long long) ctx->err_line);
      return dx_fail(ctx,DX_E_FORMAT,"Line %lld: incomplete last entry of .quiv file",
                     (long long) ctx->err_line);
    }
  const int64_t nent = nlines / 6;
  const size_t need = round_up((size_t) nent*8,256)*2 + round_up((size_t) nent*4,256)*7 + 256;
  if (ctx->qv_store_cap < need)
    { if (ctx->qv_store) cudaFree(ctx->qv_store);
      ctx->qv_store = NULL; ctx->qv_store_cap = 0;
      if (cudaMalloc((void **) &ctx->qv_store,need) != cudaSuccess)
        { ctx->qv_store = NULL; cudaGetLastError();
          return dx_fail(ctx,DX_E_NOMEM,"device allocation of %zu bytes (entry table) failed",need);
        }
      ctx->qv_store_cap = need;
    }
  QvEntries ent;
  uint8_t *p = ctx->qv_store;
  ent.n = nent;
  ent.hdr   = (int64_t *) p; p += round_up((size_t) nent*8,256);
  ent.line0 = (int64_t *) p; p += round_up((size_t) nent*8,256);
  ent.rlen  = (int32_t *) p; p += round_up((size_t) nent*4,256);
  ent.well  = (int32_t *) p; p += round_up((size_t) nent*4,256);
  ent.beg   = (int32_t *) p; p += round_up((size_t) nent*4,256);
  ent.end   = (int32_t *) p; p += round_up((size_t) nent*4,256);
  ent.qv    = (int32_t *) p; p += round_up((size_t) nent*4,256);
  ent.flag  = (int32_t *) p; p += round_up((size_t) nent*4,256);
  ent.order = (int32_t *) p;

  int32_t err[2];
  int64_t noncanon = 0, last = -1;
  if ((rc = dxk_qv_entries(ctx,d_text,n,d_nl,nlines,ent,err,totchar,&noncanon,&last)) != DX_OK) return rc;
  if (last != (int64_t) n - 1)
    { ctx->err_line = ctx->origin_line + nlines + 1;
      return dx_fail(ctx,DX_E_FORMAT,"Line %lld: Last line does not end with a newline !",
                     (long long) ctx->err_line);
    }
  if (err[0] != 0)
    { const long long line = (long long) (ctx->err_line = ctx->origin_line + err[1]);
      if (err[0] == 5)
        return dx_fail(ctx,DX_E_LINELEN,"Line %lld: Lines for an entry are not the same length",line);
      if (err[0] == 6)
        return dx_fail(ctx,DX_E_TOOLONG,"Line %lld: entry longer than 2^24 symbols",line);
      return dx_fail(ctx,DX_E_FORMAT,"Line %lld: Header in quiva file is missing",line);
    }

  // headers the device parser did not recognise as canonical: the host's sscanf decides
  std::vector<int32_t> flag;
  if (noncanon > 0 && (rc = download(ctx,ent.flag,(size_t) nent,flag)) != DX_OK) return rc;
  for (int64_t e = 0; e < nent && noncanon > 0; e++)
    { if (!flag[e]) continue;
      int64_t h0 = 0;
      DX_CUDA(ctx,cudaMemcpyAsync(&h0,ent.hdr+e,8,cudaMemcpyDeviceToHost,ctx->stream));
      DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
      std::vector<uint8_t> line;
      if ((rc = peek(ctx,d_text,n,(size_t) h0,4096,line)) != DX_OK) return rc;
      std::vector<char> txt(line.begin(),line.end());
      txt.push_back('\0');
      char *e1 = (char *) memchr(txt.data(),'\n',line.size());
      if (e1 != NULL) e1[1] = '\0';
      char *sl = strchr(txt.data()+1,'/');
      int well, beg, en, qv;
      if (sl == NULL || sscanf(sl+1,"%d/%d_%d RQ=0.%d\n",&well,&beg,&en,&qv) != 4)   // QV.c:958-968
        { ctx->err_line = ctx->origin_line + 6*e + 1;
          return dx_fail(ctx,DX_E_FORMAT,"Line %lld: Header line incorrectly formatted ?",
                         (long long) ctx->err_line);
        }
      if ((rc = upload(ctx,ent.well+e,&well,1)) != DX_OK) return rc;
      if ((rc = upload(ctx,ent.beg+e,&beg,1)) != DX_OK) return rc;
      if ((rc = upload(ctx,ent.end+e,&en,1)) != DX_OK) return rc;
      if ((rc = upload(ctx,ent.qv+e,&qv,1)) != DX_OK) return rc;
    }
  if ((rc = dxk_ticket_order(ctx,ent.rlen,nent,ent.order)) != DX_OK) return rc;
  ctx->qv_text = d_text; ctx->qv_n = n; ctx->qv_ent = ent;
  return DX_OK;
}

extern "C" int dx_qv_scan_dev(dx_ctx *ctx, const uint8_t *d_text, size_t n, const dx_qv_carry *carry,
                              dx_qv_stats *stats)
{ if (ctx == NULL || stats == NULL) return DX_E_ARG;
  int rc;
  ctx->err_line = 0;
  if ((rc = check_buf(ctx,d_text,"text")) != DX_OK) return rc;
  cudaSetDevice(ctx->device);
  dx_arena_reset(ctx);
  dx_qv_carry zero;
  if (carry == NULL)
    { memset(&zero,0,sizeof(zero));
      zero.delchar = zero.subchar = -1;
      carry = &zero;
    }
  memset(stats,0,sizeof(*stats));
  uint64_t tot = 0;
  if ((rc = qv_frame(ctx,d_text,n,&tot)) != DX_OK) return rc;
  QvProbe probe;
  if ((rc = dxk_qv_probe(ctx,d_text,ctx->qv_ent,carry,&probe)) != DX_OK) return rc;
  if ((rc = dxk_qv_hist(ctx,d_text,ctx->qv_ent,&probe,&stats->hist[0][0],NULL)) != DX_OK) return rc;

  // the kernel does not count the run characters themselves: they are what is left over
  if (probe.delchar >= 0)
    { uint64_t s = 0;
      for (int k = 0; k < 256; k++) if (k != probe.delchar) s += stats->hist[0][k];
      stats->hist[0][probe.delchar] = tot - s;
    }
  if (probe.subchar >= 0)
    { uint64_t s = 0;
      for (int k = 0; k < 256; k++) if (k != probe.subchar) s += stats->hist[3][k];
      stats->hist[3][probe.subchar] = tot - s;
    }
  stats->totchar  = tot;
  stats->nentries = ctx->qv_ent.n;
  stats->delchar  = probe.delchar;
  stats->subchar  = probe.subchar;
  memcpy(stats->sub_prefix,probe.sub_prefix,sizeof(stats->sub_prefix));
  return DX_OK;
}

// ================================================================================================
//  QV coder: encode
// ================================================================================================

// Encoder tables (dx_qv_encode.cu): bits 0-4 length of the whole item, bit 5 escape, bits 8-31 the
// item's bits.  An escaped SYMBOL carries its 8-bit literal inside the item (QV.c:432-434); an
// escaped RUN LENGTH is followed by a separate 16-bit literal (QV.c:486-487).
static void pack_tables(const dx_qv_coding *c, QvEncTables *t)
{ for (int k = 0; k < 6; k++)
    { const dx_scheme &s = c->tab[k];
      const bool isrun = (k == 1 || k == 5);
      for (int x = 0; x < 256; x++)
        { const bool esc = (isrun || s.type == 2) && s.lens[x] > 0 &&
                           s.bits[x] == s.bits[255] && s.lens[x] == s.lens[255];   // QV.c:432,486
          uint32_t len  = (uint32_t) (s.lens[x] & 0x1f);
          uint32_t bits = s.bits[x] & 0xffffu;
          if (len > 16) { len = 0; bits = 0; }          // no usable code: the symbol does not occur
          if (esc && !isrun) { bits = (bits << 8) | (uint32_t) x; len += 8; }
          t->t[k][x] = len | ((uint32_t) esc << 5) | (bits << 8);
        }
    }
}

extern "C" int dx_qv_encode_dev(dx_ctx *ctx, const uint8_t *d_text, size_t n,
                                const dx_qv_coding *coding, int lossy, int32_t lwell_in,
                                uint8_t *d_out, size_t cap, size_t *out_len, int32_t *last_well,
                                int64_t *h_entry_off, int64_t max_entries)
{ if (ctx == NULL || coding == NULL || out_len == NULL) return DX_E_ARG;
  int rc;
  *out_len = 0;
  if ((rc = check_buf(ctx,d_text,"text")) != DX_OK) return rc;
  cudaSetDevice(ctx->device);
  dx_arena_reset(ctx);
  if (ctx->qv_text != d_text || ctx->qv_n != n)
    { uint64_t tot;
      if ((rc = qv_frame(ctx,d_text,n,&tot)) != DX_OK) return rc;
    }
  QvEncTables tab;
  pack_tables(coding,&tab);
  rc = dxk_qv_encode(ctx,d_text,n,ctx->qv_ent,&tab,coding->delchar,coding->subchar,lossy,lwell_in,
                     d_out,cap,out_len,last_well,h_entry_off,max_entries);
  // The framing of dx_qv_scan_dev serves ONE encode of the same buffer: a caller that refills the
  // buffer (same address, same size) and encodes again must not meet the offsets of the old text.
  ctx->qv_text = NULL; ctx->qv_n = 0;
  return rc;
}

extern "C" int dx_qv_forget(dx_ctx *ctx)
{ if (ctx == NULL) return DX_E_ARG;
  ctx->qv_text = NULL; ctx->qv_n = 0; ctx->qv_ent.n = 0;
  return DX_OK;
}

extern "C" int dx_qv_last_well(dx_ctx *ctx, int32_t *well)
{ if (ctx == NULL || well == NULL) return DX_E_ARG;
  *well = 0;
  if (ctx->qv_text == NULL || ctx->qv_ent.n == 0) return DX_OK;
  cudaSetDevice(ctx->device);
  DX_CUDA(ctx,cudaMemcpyAsync(well,ctx->qv_ent.well + (ctx->qv_ent.n - 1),4,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  return DX_OK;
}

extern "C" int dx_text_lines_dev(dx_ctx *ctx, const uint8_t *d_text, size_t n, int64_t skip,
                                 int64_t *nlines, int64_t *skip_off)
{ if (ctx == NULL || nlines == NULL || skip < 0) return DX_E_ARG;
  int rc;
  *nlines = 0;
  if (skip_off) *skip_off = (skip == 0) ? 0 : -1;
  if (n == 0) return DX_OK;
  if ((rc = check_buf(ctx,d_text,"text")) != DX_OK) return rc;
  cudaSetDevice(ctx->device);
  dx_arena_reset(ctx);
  int64_t *d_nl = NULL, cnt = 0;
  if ((rc = dxk_index_positions(ctx,DX_PRED_NEWLINE,d_text,n,0,&d_nl,&cnt)) != DX_OK) return rc;
  *nlines = cnt;
  if (skip_off != NULL && skip > 0 && skip <= cnt)
    { int64_t at = -1;
      DX_CUDA(ctx,cudaMemcpyAsync(&at,d_nl + (skip - 1),8,cudaMemcpyDeviceToHost,ctx->stream));
      DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
      *skip_off = at + 1;
    }
  return DX_OK;
}

extern "C" int dx_dexqv_dev(dx_ctx *ctx, const uint8_t *d_text, size_t n, int lossy,
                            uint8_t *d_out, size_t cap, size_t *out_len)
{ if (ctx == NULL || out_len == NULL) return DX_E_ARG;
  int rc;
  *out_len = 0;
  dx_qv_stats  *st = (dx_qv_stats *) malloc(sizeof(dx_qv_stats));
  dx_qv_coding *cd = (dx_qv_coding *) malloc(sizeof(dx_qv_coding));
  std::vector<uint8_t> head, fh(2 + 16384 + 100000);
  size_t hlen = 0, body = 0;
  if (st == NULL || cd == NULL) { rc = DX_E_NOMEM; goto done; }
  if ((rc = dx_qv_scan_dev(ctx,d_text,n,NULL,st)) != DX_OK) goto done;
  if (st->nentries == 0) { rc = dx_fail(ctx,DX_E_FORMAT,"no entries in .quiva input"); goto done; }
  if ((rc = dx_qv_make_coding(st,lossy,cd)) != DX_OK)
    { dx_fail(ctx,rc,"a QV stream has fewer than two distinct symbols: cannot build a code");
      goto done;
    }
  // prefix := first header up to the first '/' after the '@' (dexqv.c:88-103)
  if ((rc = peek(ctx,d_text,n,0,100000,head)) != DX_OK) goto done;
  { const uint8_t *sl = (const uint8_t *) memchr(head.data()+1,'/',head.size()-1);
    if (sl == NULL) { rc = dx_fail(ctx,DX_E_FORMAT,"Header line incorrectly formatted ?"); goto done; }
    const uint16_t key = 0x55aa;                                         // dexqv.c:105-106
    memcpy(fh.data(),&key,2);
    if ((rc = dx_qv_write_coding(cd,(const char *) head.data(),(int) (sl - head.data()),
                                 fh.data()+2,fh.size()-2,&hlen)) != DX_OK)
      { dx_fail(ctx,rc,"could not write the coding header");
        goto done;
      }
    hlen += 2;
  }
  if (hlen > cap) { rc = dx_fail(ctx,DX_E_CAP,"output buffer too small for the coding header"); goto done; }
  if ((rc = upload(ctx,d_out,fh.data(),hlen)) != DX_OK) goto done;
  if ((rc = dx_qv_encode_dev(ctx,d_text,n,cd,lossy,0,d_out+hlen,cap-hlen,&body,NULL,NULL,0)) != DX_OK)
    { if (rc == DX_E_CAP && ctx->need_bytes > 0) ctx->need_bytes += hlen;   // the body's need: add the header
      goto done;
    }
  if ((rc = dx_sync(ctx)) != DX_OK) goto done;
  *out_len = hlen + body;
done:
  free(st); free(cd);
  return rc;
}

// ================================================================================================
//  QV coder: decode
// ================================================================================================

static void build_dec_tables(const dx_qv_coding *c, QvDecTables *t)
{ memset(t,0,sizeof(*t));
  for (int k = 0; k < 6; k++)
    { const dx_scheme &s = c->tab[k];
      t->type[k] = s.type;
      for (int i = 0; i < 256; i++)                       // ascending: 255 wins ties (QV.c:365-372)
        { t->lens[k][i] = (uint8_t) s.lens[i];
          if (s.lens[i] > 0 && s.lens[i] <= 16)
            { const uint32_t base = (s.bits[i] << (16 - s.lens[i])) & 0xffffu;
              const uint32_t span = 1u << (16 - s.lens[i]);
              memset(&t->look[k][base],i,span);
            }
        }
    }
}

// Two-level tables for the warp-per-entry decoder.  A scheme has at most 256 codes, so it never
// needs more than DX_DEC2_MAXSUB sub-tables.
static void build_dec_tables2(const dx_qv_coding *c, QvDecTables2 *t)
{ memset(t,0,sizeof(*t));
  for (int k = 0; k < 6; k++)
    { const dx_scheme &s = c->tab[k];
      int nsub = 0;
      t->type[k] = s.type;
      for (int i = 0; i < 256; i++)                       // ascending: 255 wins ties (QV.c:365-372)
        { const int len = s.lens[i];
          if (len <= 0 || len > 16) continue;
          const uint16_t val = (uint16_t) (i | (len << 8));
          if (len <= 11)
            { const uint32_t base = (s.bits[i] << (11 - len)) & 0x7ffu;
              for (uint32_t j = 0; j < (1u << (11 - len)); j++) t->prim[k][base + j] = val;
            }
          else
            { const uint32_t pre = (s.bits[i] >> (len - 11)) & 0x7ffu;
              uint16_t &pe = t->prim[k][pre];
              if (!(pe & 0x8000u))
                { pe = (uint16_t) (0x8000u | nsub);
                  nsub++;
                }
              const uint32_t idx = pe & 0x7fffu;
              const uint32_t base = (s.bits[i] << (16 - len)) & 31u;
              for (uint32_t j = 0; j < (1u << (16 - len)); j++) t->sub[k][idx*32 + base + j] = val;
            }
        }
    }
}

// 12-bit shared-memory tables for the parallel decoders.  A code of at most 12 bits owns the range
// of 12-bit windows it is a prefix of; filling the ranges in ascending symbol order resolves the
// ties of a type-2 scheme (symbols folded onto the escape share its code) exactly as the
// reference's 16-bit LUT does: 255 wins (QV.c:365-372).
static void build_dec_tables4(const dx_qv_coding *c, QvDecTables4 *t)
{ memset(t,0,sizeof(*t));
  build_dec_tables2(c,&t->t2);
  double ab[6], erun[6];
  for (int k = 0; k < 6; k++)
    { const dx_scheme &s = c->tab[k];
      const bool isrun = (k == 1 || k == 5);
      uint16_t *one = t->single[k];                        // sym | len << 8, 0 = no code of <= 12 bits
      for (int i = 0; i < 256; i++)
        { const int len = s.lens[i];
          if (len <= 0 || len > 12) continue;
          const uint32_t base = (s.bits[i] << (12 - len)) & 0xfffu;
          const uint16_t val = (uint16_t) (i | (len << 8));
          for (uint32_t j = 0; j < (1u << (12 - len)); j++) one[base + j] = val;
        }
      auto first = [&](uint32_t w16, int &sym, int &len) -> bool
        { const uint16_t e = one[w16 >> 4];
          sym = e & 0xff; len = e >> 8;
          return e != 0;
        };
      for (uint32_t p = 0; p < 4096; p++)
        { int s0, l0;
          if (!first(p << 4,s0,l0)) continue;
          if (isrun) continue;
          if (s.type == 2 && s0 == 255)
            { t->multi[k][p] = (uint32_t) (l0 + 8) | (1u << 5) | 0x80u | ((uint32_t) l0 << 8) | (255u << 16);
              continue;
            }
          int s1 = 0, l1 = 0;
          const bool two = (l0 < 12) && first(((p << l0) & 0xfffu) << 4,s1,l1) && l1 <= 12 - l0 &&
                           !(s.type == 2 && s1 == 255);
          if (two)
            t->multi[k][p] = (uint32_t) (l0 + l1) | (2u << 5) | ((uint32_t) l0 << 8) |
                             ((uint32_t) s0 << 16) | ((uint32_t) s1 << 24);
          else
            t->multi[k][p] = (uint32_t) l0 | (1u << 5) | ((uint32_t) l0 << 8) | ((uint32_t) s0 << 16);
        }
      // expected bits per item (and expected run length) under the code's own distribution
      ab[k] = 0; erun[k] = 0;
      for (int i = 0; i < 256; i++)
        { const int len = s.lens[i];
          if (len <= 0 || len > 16) continue;
          const bool folded = (i < 255 && s.lens[255] == len && s.bits[255] == s.bits[i] &&
                               (isrun || s.type == 2));
          if (folded) continue;
          const bool escape = (i == 255) && (isrun || s.type == 2);
          const double q = 1.0 / (double) (1u << len);
          ab[k]   += q * (len + (escape ? (isrun ? 16 : 8) : 0));
          erun[k] += q * (escape ? 400.0 : (double) i);
        }
    }
  for (int k = 0; k < 6; k++)
    { const dx_scheme &s = c->tab[k];
      const bool isrun = (k == 1 || k == 5);
      int n = 0;
      for (int i = 0; i < 256; i++)
        { const int len = s.lens[i];
          if (len <= 12 || len > 16) continue;
          const bool folded = (i < 255 && s.lens[255] == len && s.bits[255] == s.bits[i] &&
                               (isrun || s.type == 2));
          if (folded) continue;
          t->longs[k][n++] = (((s.bits[i] << (16 - len)) & 0xffffu) << 16) | ((uint32_t) len << 8) | (uint32_t) i;
        }
      std::sort(t->longs[k],t->longs[k] + n);
      t->nlong[k] = n;
    }
  t->abits[0] = (float) (c->delchar >= 0 ? (ab[0] + ab[1]) / (erun[1] + 1.0) : ab[0]);
  t->abits[2] = (float) ab[2];
  t->abits[3] = (float) ab[3];
  t->abits[4] = (float) (c->subchar >= 0 ? (ab[4] + ab[5]) / (erun[5] + 1.0) : ab[4]);
}

// bits a position takes at least: the shortest ins code plus the shortest mrg code (never run-length coded)
static int qv_minbits(const dx_qv_coding &c)
{ int minbits = 0;
  for (int k = 2; k <= 3; k++)
    { int mn = 32;
      for (int x = 0; x < 256; x++)
        if (c.tab[k].lens[x] > 0 && c.tab[k].lens[x] < mn) mn = c.tab[k].lens[x];
      minbits += (mn == 32) ? 0 : mn;
    }
  return minbits;
}

// A small asynchronous transfer between pinned host memory and the device on ctx->stream; by_kernel: by
// dxk_fetch, not queued behind the large copies of the pipelined host decode (see k_fetch, dx_frame.cu).
static int qv_copy(dx_ctx *ctx, bool by_kernel, void *dst, const void *src, size_t bytes)
{ if (by_kernel) return dxk_fetch(ctx,dst,src,bytes);
  if (bytes > 0) DX_CUDA(ctx,cudaMemcpyAsync(dst,src,bytes,cudaMemcpyDefault,ctx->stream));
  return DX_OK;
}

// The 12-bit decode tables of a coding, copied to d_tab4 through a temporary buffer (h4 == NULL, synchronous)
// or by qv_copy from pinned h4.
static int qv_tables4(dx_ctx *ctx, const dx_qv_coding *c, QvDecTables4 *h4, bool by_kernel, QvDecTables4 *d_tab4)
{ QvDecTables4 *h = h4 ? h4 : (QvDecTables4 *) malloc(sizeof(QvDecTables4));
  if (h == NULL) return DX_E_NOMEM;
  build_dec_tables4(c,h);
  const int rc = h4 ? qv_copy(ctx,by_kernel,d_tab4,h,sizeof(QvDecTables4)) : upload(ctx,d_tab4,h,1);
  if (h4 == NULL) free(h);
  return rc;
}

struct QvPlan
{ std::vector<QvDecEntry> ent;
  bool         v2;            // the parallel decoders (not the sequential kernels of dx_qv_decode.cu)
  QvDecTables4 *d_tab4;
  int64_t     *d_soff;        // v1 only: [count][6] device
  int64_t     *d_start;       // v2: first stream byte of every entry
  int32_t     *d_rlen;        // v2
  QvDecTables  *d_tab;
  char        *d_prefix;
  int          plen;
  dx_qv_coding coding;
  size_t       text_len;
  // entries discovered AND decoded in one pass (speculative decode into a scratch image):
  bool         spec;
  uint8_t     *d_tmp;         // the scratch image (lines only)
  size_t       tmp_n;
  std::vector<int64_t> src;   // per entry: offset of its lines in d_tmp, -1 = not decoded yet
  std::vector<int64_t> ix_fs, ix_end;   // per entry: first stream byte, first byte after the entry
};

// Ticket order for the one-warp-per-entry decoder: longest entries first (a warp decodes ~8 entries
// of a 2 GB file, so whatever is handed out last is the tail of the launch -- it should be short).
// Counting sort on rlen / 512, file order within a bucket.
static void ticket_order(const int32_t *rlen, size_t N, int32_t *order)
{ enum { kBuckets = 512 };
  size_t count[kBuckets + 1];
  memset(count,0,sizeof(count));
  auto bucket = [](int32_t rl) -> int
    { const int b = (rl <= 0) ? 0 : (int) (rl >> 9);
      return kBuckets - 1 - (b >= kBuckets ? kBuckets - 1 : b);           // descending length
    };
  for (size_t i = 0; i < N; i++) count[bucket(rlen[i]) + 1]++;
  for (int b = 0; b < kBuckets; b++) count[b+1] += count[b];
  for (size_t i = 0; i < N; i++) order[count[bucket(rlen[i])]++] = (int32_t) i;
}

// ... and the cut between the two parallel decoders: the first n_coop tickets (the longest entries)
// go to the warp-per-entry kernel, the others are decoded one entry per lane (dx_qv_decode6.cu).
// A lane walks its entry alone, ~kLaneNs per position, so the lane kernel lasts at least as long as
// its longest entry; below that bound it is limited by instruction issue (kLaneGBs of text), the
// warp kernel always is (kCoopGBs).  The cut that minimises the sum of the two launches is found on
// the 512 length buckets of the counting sort.
static int64_t ticket_plan(const dx_ctx *ctx, const int32_t *rlen, size_t N, int32_t *order)
{ enum { kBuckets = 512 };
  // measured on B200 (profiles/r02_decoders.txt): a lane needs 280 ns per position (the 60 000-position
  // entries of the 2 GB bench file keep k_qv_decode6 busy for 16.9 ms), the warp kernel decodes 460 GB/s
  const double kLaneNs = 280e-9, kLaneGBs = 1500e9, kCoopGBs = 460e9, kLaunch = 8e-6;
  ticket_order(rlen,N,order);
  const int64_t mode = ctx->route[DXR_DECODER];
  if (mode == 5 || N == 0) return (int64_t) N;
  if (mode == 6) return 0;
  static thread_local double bsum[kBuckets];
  static thread_local int64_t bcnt[kBuckets];
  for (int b = 0; b < kBuckets; b++) { bsum[b] = 0; bcnt[b] = 0; }
  double all = 0;
  for (size_t i = 0; i < N; i++)
    { const int32_t rl = rlen[i];
      const int b = (rl <= 0) ? 0 : ((rl >> 9) >= kBuckets ? kBuckets - 1 : (rl >> 9));
      bsum[b] += (rl > 0) ? 5.0*rl : 0.0; bcnt[b]++;
      all += (rl > 0) ? 5.0*rl : 0.0;
    }
  if (ctx->route[DXR_LANE_MAX_RLEN] > 0)
    { int64_t nc = 0;
      const int64_t cutb = ctx->route[DXR_LANE_MAX_RLEN] >> 9;
      for (int b = kBuckets - 1; b > cutb; b--) nc += bcnt[b];
      return nc;
    }
  // cut after bucket c: buckets > c coop, <= c lane
  double best = all / kCoopGBs + kLaunch, coop = 0;
  int64_t best_n = (int64_t) N, ncoop = 0;
  for (int c = kBuckets - 1; c >= 0; c--)
    { // lane part = buckets 0..c
      const double lane_bytes = all - coop;
      const double t_lane = std::max((double) ((c + 1) << 9) * kLaneNs,lane_bytes / kLaneGBs) + kLaunch;
      const double t = t_lane + (ncoop > 0 ? coop / kCoopGBs + kLaunch : 0.0);
      if (t < best && (int64_t) N - ncoop > 0) { best = t; best_n = ncoop; }
      coop += bsum[c]; ncoop += bcnt[c];
    }
  const int64_t minlane = ctx->route[DXR_LANE_MIN_ENTRIES] > 0 ? ctx->route[DXR_LANE_MIN_ENTRIES] : 1;
  if ((int64_t) N - best_n < minlane) return (int64_t) N;
  return best_n;
}

static int64_t lpt_order(const dx_ctx *ctx, const std::vector<CandInfo> &info, std::vector<int32_t> &order)
{ const size_t N = info.size();
  std::vector<int32_t> rl(N);
  for (size_t i = 0; i < N; i++) rl[i] = le32(info[i].field+4) - le32(info[i].field);
  order.resize(N);
  return ticket_plan(ctx,rl.data(),N,order.data());
}

struct QvWalkUser
{ const uint8_t *d_in; size_t n; const QvPlan *plan;
  std::vector<int64_t> side;           // 6 stream offsets per slow-path entry
  int fieldbytes;                      // 12: int32 beg/end/qv; 6: the old layout's uint16 (undexqv.c:162-180)
  int flip;                            // fields (and stream words) in the other byte order
};

// field k (0 beg, 1 end, 2 qv) of an entry header in either layout and byte order (undexqv.c:135-180)
static int32_t qv_field(const uint8_t *f, int k, int fieldbytes, int flip)
{ if (fieldbytes == 12)
    { const uint8_t *p = f + 4*k;
      return flip ? (int32_t) ((uint32_t) p[3] | ((uint32_t) p[2] << 8) | ((uint32_t) p[1] << 16) | ((uint32_t) p[0] << 24))
                  : le32(p);
    }
  const uint8_t *p = f + 2*k;
  return flip ? (int32_t) ((uint32_t) p[1] | ((uint32_t) p[0] << 8)) : (int32_t) ((uint32_t) p[0] | ((uint32_t) p[1] << 8));
}

// walk `count` entries whose first stream byte / length are on the device
static int qv_walk(dx_ctx *ctx, const uint8_t *d_in, size_t n, const QvPlan &plan,
                   const int64_t *d_start, const int32_t *d_rlen, int64_t count,
                   int64_t *d_soff, int32_t *d_stat)
{ const dx_qv_coding &cd = plan.coding;
  if (plan.v2)
    return dxk_qv_decode5(ctx,d_in,n,plan.d_tab4,cd.delchar,cd.subchar,0,0,count,d_start,d_rlen,
                          NULL,NULL,0,NULL,d_soff,d_stat);
  return dxk_qv_walk(ctx,d_in,n,plan.d_tab,cd.delchar,cd.subchar,cd.flip,d_start,d_rlen,count,
                     d_soff,d_stat);
}

static int qv_walk_one(dx_ctx *ctx, void *user, int64_t q, int64_t *end, int64_t *slot)
{ QvWalkUser *u = (QvWalkUser *) user;
  int rc;
  std::vector<uint8_t> f;
  const int fb = u->fieldbytes;
  if ((rc = peek(ctx,u->d_in,u->n,(size_t) q,(size_t) fb,f)) != DX_OK) return rc;
  *slot = (int64_t) (u->side.size() / 6);
  if ((int) f.size() < fb) { *end = -1; return DX_OK; }
  const int32_t rlen = qv_field(f.data(),1,fb,u->flip) - qv_field(f.data(),0,fb,u->flip);
  if (rlen < 0) return dx_fail(ctx,DX_E_FORMAT,"negative read length in entry header");
  if (rlen >= (1 << 24)) { *end = -1; return DX_OK; }
  int64_t *d_start = (int64_t *) dx_arena_get(ctx,8);
  int32_t *d_rlen  = (int32_t *) dx_arena_get(ctx,4);
  int64_t *d_soff  = (int64_t *) dx_arena_get(ctx,48);
  int32_t *d_stat  = (int32_t *) dx_arena_get(ctx,4);
  if (!d_start || !d_rlen || !d_soff || !d_stat) return DX_E_NOMEM;
  const int64_t start = q + fb;
  if ((rc = upload(ctx,d_start,&start,1)) != DX_OK) return rc;
  if ((rc = upload(ctx,d_rlen,&rlen,1)) != DX_OK) return rc;
  if ((rc = qv_walk(ctx,u->d_in,u->n,*u->plan,d_start,d_rlen,1,d_soff,d_stat)) != DX_OK) return rc;
  std::vector<int64_t> so; std::vector<int32_t> stt;
  if ((rc = download(ctx,d_soff,6,so)) != DX_OK) return rc;
  if ((rc = download(ctx,d_stat,1,stt)) != DX_OK) return rc;
  *end = stt[0] ? -1 : so[5];
  u->side.insert(u->side.end(),so.begin(),so.end());
  return DX_OK;
}

// The head of a .dexqv image, read from host bytes.  New layout: 0x55aa (either byte order) in front
// of the coding header; old layout: the file starts with the coding header itself (key 0x33cc) and
// beg/end/qv are uint16 (undexqv.c:103-110).
struct QvHead
{ uint16_t          key;
  bool              newv;         // the new layout
  dx_qv_coding      coding;
  std::vector<char> prefix = std::vector<char>(100001);   // NUL-terminated
  int               plen;
  size_t            first;        // first byte behind the coding header
};

// DX_E_TRUNC: fewer than 2 bytes; DX_E_KEY: no .dexqv key; else what dx_qv_read_coding returns.  No
// message: the fast paths decline such an image silently, the general path says what is wrong.
static int qv_read_head(const uint8_t *h, size_t len, QvHead &hd)
{ if (len < 2) return DX_E_TRUNC;
  memcpy(&hd.key,h,2);
  hd.newv = (hd.key == 0x55aa || hd.key == 0xaa55);
  if (!hd.newv && !(hd.key == 0x33cc || hd.key == 0xcc33)) return DX_E_KEY;
  const size_t keylen = hd.newv ? 2 : 0;
  size_t used = 0;
  const int rc = dx_qv_read_coding(h + keylen,len - keylen,&hd.coding,hd.prefix.data(),(int) hd.prefix.size(),&used);
  if (rc != DX_OK) return rc;
  hd.plen = (int) strlen(hd.prefix.data());
  hd.first = keylen + used;
  return DX_OK;
}

static int plan_undexqv(dx_ctx *ctx, const uint8_t *d_in, size_t n, const int64_t *h_entry_off,
                        int64_t nentries, int32_t well_in, bool need_streams, int upper, QvPlan &plan)
{ int rc;
  std::vector<uint8_t> head;
  if ((rc = peek(ctx,d_in,n,0,2 + 16384 + 100000,head)) != DX_OK) return rc;
  if (head.size() < 2) return dx_fail(ctx,DX_E_TRUNC,"System error, read failed!");
  QvHead hd;
  if ((rc = qv_read_head(head.data(),head.size(),hd)) == DX_E_KEY)
    return dx_fail(ctx,DX_E_KEY,"not a .dexqv file (endian key 0x%04x)",(unsigned) hd.key);
  if (rc != DX_OK) return dx_fail(ctx,rc,"Could not read the coding header (Read_QVcoding)");
  plan.coding = hd.coding;
  // A file of the other byte order (every stream word flipped, QV.c:553-568) or of the old layout is
  // rare: it takes the sequential kernels, which flip words as they read them, and finds its
  // entries by walking them one after the other.  Slow (a launch per entry), but the reference's bytes.
  const bool legacy = (plan.coding.flip != 0) || !hd.newv;
  const int fieldbytes = hd.newv ? 12 : 6;
  if (legacy) { h_entry_off = NULL; nentries = 0; }
  const size_t first = hd.first;
  DxPhases ph(ctx);
  plan.plen = hd.plen;
  plan.d_soff = NULL; plan.d_start = NULL; plan.d_rlen = NULL; plan.d_tab = NULL;
  plan.spec = false; plan.d_tmp = NULL; plan.tmp_n = 0; plan.src.clear();

  plan.v2 = (ctx->route[DXR_DECODER] != 1 && !legacy);
  plan.d_tab4 = NULL;
  if (plan.v2)
    { if ((plan.d_tab4 = (QvDecTables4 *) dx_arena_get(ctx,sizeof(QvDecTables4))) == NULL) return DX_E_NOMEM;
      if ((rc = qv_tables4(ctx,&plan.coding,NULL,false,plan.d_tab4)) != DX_OK) return rc;
    }
  if (!plan.v2)
    { QvDecTables *h_tab = (QvDecTables *) malloc(sizeof(QvDecTables));
      if (h_tab == NULL) return DX_E_NOMEM;
      build_dec_tables(&plan.coding,h_tab);
      plan.d_tab = (QvDecTables *) dx_arena_get(ctx,sizeof(QvDecTables));
      rc = plan.d_tab ? upload(ctx,plan.d_tab,h_tab,1) : DX_E_NOMEM;
      free(h_tab);
      if (rc != DX_OK) return rc;
    }
  plan.d_prefix = (char *) dx_arena_get(ctx,(size_t) plan.plen + 1);
  if (!plan.d_prefix) return DX_E_NOMEM;
  if ((rc = upload(ctx,plan.d_prefix,hd.prefix.data(),(size_t) plan.plen)) != DX_OK) return rc;

  struct Hdr { int32_t well, beg, end, qv; };
  std::vector<Hdr> hdrs;
  const bool want_soff = need_streams && !plan.v2;      // v1 decode kernel needs stream offsets

  if (h_entry_off != NULL)
    { // entry starts are known (our encoder's index, or Dazzler .idx coff, DB.c:2598)
      const size_t N = (size_t) nentries;
      int64_t  *d_estart = (int64_t *) dx_arena_get(ctx,N*8);
      int64_t  *d_q      = (int64_t *) dx_arena_get(ctx,N*8);
      CandInfo *d_info   = (CandInfo *) dx_arena_get(ctx,N*sizeof(CandInfo));
      plan.d_start       = (int64_t *) dx_arena_get(ctx,N*8);
      plan.d_rlen        = (int32_t *) dx_arena_get(ctx,N*4);
      if (!d_estart || !d_q || !d_info || !plan.d_start || !plan.d_rlen) return DX_E_NOMEM;
      if ((rc = upload(ctx,d_estart,h_entry_off,N)) != DX_OK) return rc;
      if ((rc = dxk_skip_ff(ctx,d_in,n,d_estart,(int64_t) N,d_q)) != DX_OK) return rc;
      if ((rc = dxk_field_rlen(ctx,d_in,d_q,(int64_t) N,plan.d_rlen)) != DX_OK) return rc;
      if ((rc = dxk_cand_context(ctx,d_in,n,first,d_q,(int64_t) N,12,d_info)) != DX_OK) return rc;
      std::vector<int64_t> q;
      if ((rc = download(ctx,d_q,N,q)) != DX_OK) return rc;
      std::vector<int64_t> fs(N);
      for (size_t i = 0; i < N; i++) fs[i] = q[i] + 12;
      if ((rc = upload(ctx,plan.d_start,fs.data(),N)) != DX_OK) return rc;
      std::vector<CandInfo> info;
      if ((rc = download(ctx,d_info,N,info)) != DX_OK) return rc;
      if (want_soff)
        { int32_t *d_stat = (int32_t *) dx_arena_get(ctx,N*4);
          plan.d_soff = (int64_t *) dx_arena_get(ctx,N*48);
          if (!d_stat || !plan.d_soff) return DX_E_NOMEM;
          if ((rc = qv_walk(ctx,d_in,n,plan,plan.d_start,plan.d_rlen,(int64_t) N,plan.d_soff,d_stat)) != DX_OK)
            return rc;
          std::vector<int32_t> stat;
          if ((rc = download(ctx,d_stat,N,stat)) != DX_OK) return rc;
          for (size_t i = 0; i < N; i++)
            if (stat[i]) return dx_fail(ctx,DX_E_TRUNC,"Could not read more bits (Decode), entry %zu",i+1);
          std::vector<int64_t> soff;                            // entry i must end where entry i+1 starts
          if ((rc = download(ctx,plan.d_soff,N*6,soff)) != DX_OK) return rc;
          for (size_t i = 0; i < N; i++)
            if (soff[6*i+5] != ((i + 1 < N) ? h_entry_off[i+1] : (int64_t) n))
              return dx_fail(ctx,DX_E_FORMAT,"entry %zu: its streams do not end at the next entry",i+1);
        }
      plan.ix_fs = fs;
      plan.ix_end.resize(N);
      for (size_t i = 0; i < N; i++) plan.ix_end[i] = (i + 1 < N) ? h_entry_off[i+1] : (int64_t) n;
      int32_t well = well_in;
      hdrs.resize(N);
      for (size_t i = 0; i < N; i++)
        { well += 255 * (int32_t) (q[i] - 1 - h_entry_off[i]) + info[i].last;
          hdrs[i].well = well;
          hdrs[i].beg = le32(info[i].field); hdrs[i].end = le32(info[i].field+4);
          hdrs[i].qv  = le32(info[i].field+8);
        }
    }
  else
    { int64_t *d_q = NULL, nc = 0;
      ph.mark("tables");
      if (!legacy &&
          (rc = dxk_index_positions(ctx,DX_PRED_QVCAND,d_in,n,first + 1,&d_q,&nc)) != DX_OK) return rc;
      ph.mark("index");
      const size_t N = (size_t) nc;
      int64_t  *d_fs    = (int64_t *) dx_arena_get(ctx,N*8);
      int32_t  *d_rlen  = (int32_t *) dx_arena_get(ctx,N*4);
      int32_t  *d_stat  = (int32_t *) dx_arena_get(ctx,N*4);
      int64_t  *d_soffc = (int64_t *) dx_arena_get(ctx,N*48);
      CandInfo *d_info  = (CandInfo *) dx_arena_get(ctx,N*sizeof(CandInfo));
      if (!d_fs || !d_rlen || !d_stat || !d_soffc || !d_info) return DX_E_NOMEM;
      if ((rc = dxk_field_rlen(ctx,d_in,d_q,nc,d_rlen)) != DX_OK) return rc;
      if ((rc = dxk_cand_context(ctx,d_in,n,first,d_q,nc,12,d_info)) != DX_OK) return rc;
      std::vector<int64_t> q, fs;
      if ((rc = download(ctx,d_q,N,q)) != DX_OK) return rc;
      fs.resize(N);
      for (size_t i = 0; i < N; i++) fs[i] = q[i] + 12;
      if ((rc = upload(ctx,d_fs,fs.data(),N)) != DX_OK) return rc;
      std::vector<CandInfo> info;
      if ((rc = download(ctx,d_info,N,info)) != DX_OK) return rc;
      ph.mark("context");
      std::vector<int64_t> tmp_off(N + 1,0);
      if (need_streams && plan.v2 && !ctx->route[DXR_NO_SPEC])
        { // decode every candidate right away into a scratch image laid out by the candidates'
          // own lengths; the chain below decides which of them are entries
          for (size_t i = 0; i < N; i++)
            { int64_t rl = (int64_t) le32(info[i].field+4) - le32(info[i].field);
              if (rl < 0 || rl >= (1 << 24)) rl = 0;
              tmp_off[i+1] = tmp_off[i] + 5*(rl + 1);
            }
          plan.tmp_n = (size_t) tmp_off[N];
          plan.d_tmp = (uint8_t *) dx_arena_get(ctx,plan.tmp_n + 64);
          QvDecEntry *d_cent = (QvDecEntry *) dx_arena_get(ctx,N*sizeof(QvDecEntry));
          if (!plan.d_tmp || !d_cent) return DX_E_NOMEM;
          std::vector<QvDecEntry> cent(N);
          for (size_t i = 0; i < N; i++)
            { memset(&cent[i],0,sizeof(QvDecEntry));
              cent[i].out_off = -1; cent[i].text_off = tmp_off[i];
            }
          if ((rc = upload(ctx,d_cent,cent.data(),N)) != DX_OK) return rc;
          // A candidate that is not an entry decodes garbage for as long as its (random) length
          // field says.  Bound it: an entry may contain a few false candidates, so candidate i must
          // end before the fields of the kSpan-th candidate after it, not counting candidates
          // closer than 64 bytes to the previous counted one (clusters in zero-rich data).  An
          // entry that breaks this rule is reported bad and found again by the chain's slow path.
          const int kSpan = 4;
          std::vector<int64_t> limit(N);
          { std::vector<size_t> nextfar(N);               // next candidate >= 64 bytes further on
            size_t j = 0;
            for (size_t i = 0; i < N; i++)
              { if (j <= i) j = i + 1;
                while (j < N && q[j] - q[i] < 64) j++;
                nextfar[i] = j;
              }
            for (size_t i = 0; i < N; i++)
              { size_t k = i;
                for (int h = 0; h < kSpan && k < N; h++) k = nextfar[k];
                limit[i] = (k < N) ? q[k] : (int64_t) n;
              }
          }
          // ... and a candidate whose length field cannot fit before its limit even at the
          // shortest code of the two streams that are never run-length coded is not decoded at all
          { const int minbits = qv_minbits(plan.coding);
            std::vector<int32_t> rl;
            size_t skipped = 0;
            if ((rc = download(ctx,d_rlen,N,rl)) != DX_OK) return rc;
            for (size_t i = 0; i < N; i++)
              if (rl[i] > 0 && q[i] + 12 + (((int64_t) rl[i]*minbits) >> 3) > limit[i])
                { rl[i] = -1; skipped++; }
            if (skipped)
              if ((rc = upload(ctx,d_rlen,rl.data(),N)) != DX_OK) return rc;
            if (ctx->route[DXR_DEBUG])
              fprintf(stderr,"[dexb200 debug] undexqv: %zu of %zu candidates cannot fit (min %d bits/position)\n",
                      skipped,N,minbits);
          }
          std::vector<int32_t> order;
          const int64_t n_coop = lpt_order(ctx,info,order);
          int64_t *d_limit = (int64_t *) dx_arena_get(ctx,N*8);
          int32_t *d_order = (int32_t *) dx_arena_get(ctx,N*4);
          if (!d_limit || !d_order) return DX_E_NOMEM;
          if ((rc = upload(ctx,d_limit,limit.data(),N)) != DX_OK) return rc;
          if ((rc = upload(ctx,d_order,order.data(),N)) != DX_OK) return rc;
          const dx_qv_coding &cd = plan.coding;
          if ((rc = dxk_qv_decode6x(ctx,d_in,n,plan.d_tab4,cd.delchar,cd.subchar,upper,2,nc,d_fs,d_rlen,
                                    d_cent,NULL,0,plan.d_tmp,d_soffc,d_stat,d_limit,d_order,NULL,n_coop)) != DX_OK) return rc;
          plan.spec = true;
        }
      else if ((rc = qv_walk(ctx,d_in,n,plan,d_fs,d_rlen,nc,d_soffc,d_stat)) != DX_OK) return rc;
      ph.mark("launch");
      std::vector<int64_t> soff;
      std::vector<int32_t> stat;
      if ((rc = download(ctx,d_soffc,N*6,soff)) != DX_OK) return rc;
      if ((rc = download(ctx,d_stat,N,stat)) != DX_OK) return rc;
      ph.mark("decode+download");
      std::vector<int64_t> end(N);
      for (size_t i = 0; i < N; i++) end[i] = stat[i] ? -1 : soff[6*i+5];
      QvWalkUser user = { d_in, n, &plan, {}, fieldbytes, plan.coding.flip };
      std::vector<ChainEntry> chain;
      if ((rc = resolve_chain(ctx,d_in,n,first,fieldbytes,q,end,info,qv_walk_one,&user,chain)) != DX_OK)
        return rc;
      ph.mark("chain");
      const size_t M = chain.size();
      if (ctx->route[DXR_DEBUG])
        { int64_t sumrl = 0, maxrl = 0;
          for (size_t i = 0; i < N; i++)
            { const int64_t rl = (int64_t) le32(info[i].field+4) - le32(info[i].field);
              sumrl += rl; if (rl > maxrl) maxrl = rl;
            }
          fprintf(stderr,"[dexb200 debug] undexqv: %zu candidates (sum rlen %lld, max %lld), %zu entries, spec %d\n",
                  N,(long long) sumrl,(long long) maxrl,M,(int) plan.spec);
        }
      std::vector<int64_t> so(M*6), st(M);
      std::vector<int32_t> rl(M);
      hdrs.resize(M);
      if (plan.spec) plan.src.resize(M);
      for (size_t i = 0; i < M; i++)
        { const ChainEntry &c = chain[i];
          if (plan.spec) plan.src[i] = (c.cand >= 0) ? tmp_off[(size_t) c.cand] : -1;
          const int64_t *src = (c.cand >= 0) ? &soff[6*(size_t) c.cand]
                                             : &user.side[6*(size_t) (-2 - c.cand)];
          memcpy(&so[6*i],src,48);
          hdrs[i].well = c.well + well_in;
          hdrs[i].beg = qv_field(c.field,0,fieldbytes,plan.coding.flip);
          hdrs[i].end = qv_field(c.field,1,fieldbytes,plan.coding.flip);
          hdrs[i].qv  = qv_field(c.field,2,fieldbytes,plan.coding.flip);
          st[i] = c.q + fieldbytes;
          rl[i] = hdrs[i].end - hdrs[i].beg;
        }
      plan.ix_fs = st;
      plan.ix_end.resize(M);
      for (size_t i = 0; i < M; i++) plan.ix_end[i] = chain[i].end;
      if (need_streams)
        { plan.d_start = (int64_t *) dx_arena_get(ctx,M*8);
          plan.d_rlen  = (int32_t *) dx_arena_get(ctx,M*4);
          if (!plan.d_start || !plan.d_rlen) return DX_E_NOMEM;
          if ((rc = upload(ctx,plan.d_start,st.data(),M)) != DX_OK) return rc;
          if ((rc = upload(ctx,plan.d_rlen,rl.data(),M)) != DX_OK) return rc;
          if (want_soff)
            { plan.d_soff = (int64_t *) dx_arena_get(ctx,M*48);
              if (!plan.d_soff) return DX_E_NOMEM;
              if ((rc = upload(ctx,plan.d_soff,so.data(),M*6)) != DX_OK) return rc;
            }
        }
    }

  // output layout (undexqv.c:182, 206-207)
  size_t at = 0;
  plan.ent.resize(hdrs.size());
  for (size_t i = 0; i < hdrs.size(); i++)
    { QvDecEntry &d = plan.ent[i];
      const Hdr &h = hdrs[i];
      d.well = h.well; d.beg = h.beg; d.end = h.end; d.qv = h.qv;
      d.out_off = (int64_t) at;
      at += (size_t) plan.plen + 1 + ndigits(h.well) + 1 + ndigits(h.beg) + 1 + ndigits(h.end)
          + 6 + ndigits(h.qv) + 1;
      d.text_off = (int64_t) at;
      const int64_t rlen = (int64_t) h.end - h.beg;
      if (rlen < 0 || rlen >= (1 << 24))
        return dx_fail(ctx,DX_E_FORMAT,"unusable read length %lld in entry header",(long long) rlen);
      at += (size_t) (5*(rlen + 1));
    }
  plan.text_len = at;
  ph.mark("layout");
  ph.report("plan_undexqv");
  return DX_OK;
}

// pinned landing place of a byte total and a flag that a planning step hands back to the host
struct QvTail { int64_t total; int32_t flag; int32_t pad; };

static bool alloc_plan(dx_ctx *ctx, size_t N, QvPlanArrays &pa)
{ pa.fs    = (int64_t *)  dx_arena_get(ctx,N*8);
  pa.rlen  = (int32_t *)  dx_arena_get(ctx,N*4);
  pa.delta = (uint32_t *) dx_arena_get(ctx,N*4);
  pa.beg   = (int32_t *)  dx_arena_get(ctx,N*4);
  pa.end   = (int32_t *)  dx_arena_get(ctx,N*4);
  pa.qv    = (int32_t *)  dx_arena_get(ctx,N*4);
  return pa.fs && pa.rlen && pa.delta && pa.beg && pa.end && pa.qv;
}

// ------------------------------------------------------------------------------------------------
//  Discovered entries, for undexqv_fast (a whole image) and undexqv_pipe (one window at a time), in
//  the order a caller runs the steps: qv_cands_prep enqueues the candidates' context and limits,
//  qv_cands_plan brings what the ticket plan needs to the host, qv_cands_decode decodes every
//  candidate into a scratch image laid out by the candidates' own lengths; with their ends on the
//  host dx_chain_walk picks the entries (h_cand / h_well), qv_layout lays out their text, and the
//  caller checks its size and moves the lines into place (k_qv_assemble).  by_kernel: the small
//  transfers go through dxk_fetch (qv_copy).
// ------------------------------------------------------------------------------------------------
struct QvCands
{ size_t       N;
  const int64_t *d_q;                     // the candidates' field positions
  QvTail      *h_tail;
  QvPlanArrays pa;
  uint32_t    *d_tlen;
  int64_t     *d_limit, *d_toff, *d_soff, *h_q, *h_soff;
  int32_t     *d_ffrun, *d_stat, *d_order, *h_ffrun, *h_rlen, *h_order, *h_stat;
  uint8_t     *d_last, *h_last;
  int32_t     *h_cand, *h_well;           // the chain: entry m is candidate h_cand[m], of well h_well[m]
  int64_t      n_coop;
  uint8_t     *d_tmp;                     // the scratch image
  size_t       tmp_n;
  QvDecEntry  *d_ent;                     // qv_layout: the entries' table and where their lines are in d_tmp
  int64_t     *d_src;
};

static int qv_cands_prep(dx_ctx *ctx, const uint8_t *d_in, size_t n, size_t first, const int64_t *d_q, int64_t nc,
                         int minbits, QvTail *h_tail, QvCands &c)
{ const size_t N = (size_t) nc;
  c.N = N; c.d_q = d_q; c.h_tail = h_tail;
  c.d_tlen  = (uint32_t *) dx_arena_get(ctx,N*4);
  c.d_limit = (int64_t *)  dx_arena_get(ctx,N*8);
  c.d_ffrun = (int32_t *)  dx_arena_get(ctx,N*4);
  c.d_last  = (uint8_t *)  dx_arena_get(ctx,N);
  c.d_toff  = (int64_t *)  dx_arena_get(ctx,(N+1)*8);
  c.d_soff  = (int64_t *)  dx_arena_get(ctx,N*48);
  c.d_stat  = (int32_t *)  dx_arena_get(ctx,N*4);
  c.d_order = (int32_t *)  dx_arena_get(ctx,N*4);
  c.h_q     = (int64_t *)  dx_hpin_get(ctx,N*8);
  c.h_ffrun = (int32_t *)  dx_hpin_get(ctx,N*4);
  c.h_last  = (uint8_t *)  dx_hpin_get(ctx,N);
  c.h_rlen  = (int32_t *)  dx_hpin_get(ctx,N*4);
  c.h_order = (int32_t *)  dx_hpin_get(ctx,N*4);
  c.h_soff  = (int64_t *)  dx_hpin_get(ctx,N*48);
  c.h_stat  = (int32_t *)  dx_hpin_get(ctx,N*4);
  c.h_cand  = (int32_t *)  dx_hpin_get(ctx,N*4);
  c.h_well  = (int32_t *)  dx_hpin_get(ctx,N*4);
  if (!alloc_plan(ctx,N,c.pa) || !c.d_tlen || !c.d_limit || !c.d_ffrun || !c.d_last || !c.d_toff || !c.d_soff ||
      !c.d_stat || !c.d_order || !c.h_q || !c.h_ffrun || !c.h_last || !c.h_rlen || !c.h_order || !c.h_soff ||
      !c.h_stat || !c.h_cand || !c.h_well) return DX_E_NOMEM;
  const int rc = dxk_qv_cand_prep(ctx,d_in,n,first,d_q,nc,4,minbits,c.pa,c.d_tlen,c.d_limit,c.d_ffrun,c.d_last);
  return (rc != DX_OK) ? rc : dxk_scan_u32(ctx,c.d_tlen,nc,c.d_toff);
}

// (the synchronisation also covers whatever the caller enqueued after qv_cands_prep)
static int qv_cands_plan(dx_ctx *ctx, QvCands &c, bool by_kernel)
{ const size_t N = c.N;
  int rc;
  if ((rc = qv_copy(ctx,by_kernel,c.h_q,c.d_q,N*8)) != DX_OK ||
      (rc = qv_copy(ctx,by_kernel,c.h_ffrun,c.d_ffrun,N*4)) != DX_OK ||
      (rc = qv_copy(ctx,by_kernel,c.h_last,c.d_last,N)) != DX_OK ||
      (rc = qv_copy(ctx,by_kernel,c.h_rlen,c.pa.rlen,N*4)) != DX_OK ||
      (rc = qv_copy(ctx,by_kernel,&c.h_tail->total,c.d_toff+N,8)) != DX_OK) return rc;
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  c.tmp_n = (size_t) c.h_tail->total;
  c.n_coop = ticket_plan(ctx,c.h_rlen,N,c.h_order);
  return qv_copy(ctx,by_kernel,c.d_order,c.h_order,N*4);
}

static int qv_cands_decode(dx_ctx *ctx, const uint8_t *d_in, size_t n, const QvDecTables4 *d_tab4,
                           const dx_qv_coding &cd, int upper, QvCands &c)
{ c.d_tmp = (uint8_t *) dx_arena_get(ctx,c.tmp_n + 64);
  if (c.d_tmp == NULL) return DX_E_NOMEM;
  return dxk_qv_decode6x(ctx,d_in,n,d_tab4,cd.delchar,cd.subchar,upper,2,(int64_t) c.N,c.pa.fs,c.pa.rlen,NULL,NULL,0,
                         c.d_tmp,c.d_soff,c.d_stat,c.d_limit,c.d_order,c.d_toff,c.n_coop);
}

// the text layout of the chain's M entries; *total: its bytes (d_flag[0], zero on entry: unusable read length)
static int qv_layout(dx_ctx *ctx, QvCands &c, size_t M, int plen, int32_t *d_flag, bool by_kernel, size_t *total)
{ int32_t *d_cand  = (int32_t *) dx_arena_get(ctx,M*4 + 4);
  int32_t *d_wells = (int32_t *) dx_arena_get(ctx,M*4 + 4);
  int32_t *d_well  = (int32_t *) dx_arena_get(ctx,M*4 + 4);
  uint32_t *d_len  = (uint32_t *) dx_arena_get(ctx,M*4 + 4);
  int64_t *d_opre  = (int64_t *) dx_arena_get(ctx,(M+1)*8);
  c.d_src = (int64_t *) dx_arena_get(ctx,M*8 + 8);
  c.d_ent = (QvDecEntry *) dx_arena_get(ctx,(M+1)*sizeof(QvDecEntry));
  if (!d_cand || !d_wells || !d_well || !d_len || !d_opre || !c.d_src || !c.d_ent) return DX_E_NOMEM;
  int rc;
  if ((rc = qv_copy(ctx,by_kernel,d_cand,c.h_cand,M*4)) != DX_OK ||
      (rc = qv_copy(ctx,by_kernel,d_wells,c.h_well,M*4)) != DX_OK ||
      (rc = dxk_qv_text_len(ctx,(int64_t) M,d_cand,c.pa,NULL,d_wells,0,plen,d_len,d_well,d_flag)) != DX_OK ||
      (rc = dxk_scan_u32(ctx,d_len,(int64_t) M,d_opre)) != DX_OK ||
      (rc = dxk_qv_build_ent(ctx,(int64_t) M,d_cand,c.pa,d_well,d_opre,d_len,c.d_toff,c.d_ent,c.d_src,NULL,NULL)) != DX_OK ||
      (rc = qv_copy(ctx,by_kernel,&c.h_tail->total,d_opre+M,8)) != DX_OK ||
      (rc = qv_copy(ctx,by_kernel,&c.h_tail->flag,d_flag,4)) != DX_OK) return rc;
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  if (c.h_tail->flag) return dx_fail(ctx,DX_E_FORMAT,"unusable read length in an entry header");
  *total = (size_t) c.h_tail->total;
  return DX_OK;
}

// ctx->last_index (dx_keep_index): entry i's table row, first stream byte and first byte behind it
static void set_last_index(dx_ctx *ctx, size_t N, const QvDecEntry *ent, const int64_t *stream_off,
                           const int64_t *end_off)
{ std::vector<dx_index_row> &ix = *(std::vector<dx_index_row> *) ctx->last_index;
  ix.resize(N);
  for (size_t i = 0; i < N; i++)
    { ix[i].stream_off = stream_off[i]; ix[i].end_off = end_off[i];
      ix[i].text_off = ent[i].text_off; ix[i].rlen = ent[i].end - ent[i].beg; ix[i].well = ent[i].well;
    }
}

// ------------------------------------------------------------------------------------------------
//  The usual case of dx_undexqv_dev with everything but the verification of the entry chain on the
//  device (dx_qv_plan.cu): well numbers and text offsets are prefix sums, the host sees a few
//  bytes per entry through pinned memory.  Returns *handled = false (nothing written) when the
//  file needs the general path below: an entry the candidate filter missed.
// ------------------------------------------------------------------------------------------------
static int undexqv_fast(dx_ctx *ctx, const uint8_t *d_in, size_t n, int upper, uint8_t *d_out, size_t cap,
                        size_t *out_len, const int64_t *h_entry_off, int64_t nentries, int32_t well_in,
                        bool *handled)
{ int rc;
  *handled = false;
  DxPhases ph(ctx);
  if (ctx->route[DXR_DECODER] == 1 || ctx->route[DXR_NO_SPEC] || ctx->route[DXR_NO_FAST]) return DX_OK;
  std::vector<uint8_t> head;
  if ((rc = peek(ctx,d_in,n,0,2 + 16384 + 100000,head)) != DX_OK) return rc;
  QvHead hd;
  if (qv_read_head(head.data(),head.size(),hd) != DX_OK || !hd.newv || hd.coding.flip) return DX_OK;
  const dx_qv_coding &coding = hd.coding;
  const size_t first = hd.first;
  const int plen = hd.plen;
  QvDecTables4 *h4 = (QvDecTables4 *) dx_hpin_get(ctx,sizeof(QvDecTables4));
  if (h4 == NULL) return DX_E_NOMEM;
  QvDecTables4 *d_tab4 = (QvDecTables4 *) dx_arena_get(ctx,sizeof(QvDecTables4));
  char *d_prefix = (char *) dx_arena_get(ctx,(size_t) plen + 1);
  int32_t *d_flag = (int32_t *) dx_arena_get(ctx,16);
  if (!d_tab4 || !d_prefix || !d_flag) return DX_E_NOMEM;
  // the decode tables are host work (~0.1 ms): with a known entry index they are built while the
  // planning kernels run
  auto make_tables = [&]() -> int { return qv_tables4(ctx,&coding,h4,false,d_tab4); };
  // ... and while the candidate index runs when there is none
  struct Deferred { decltype(make_tables) *fn; int rc; } deferred = { &make_tables, DX_OK };
  char *h_prefix = (char *) dx_hpin_get(ctx,(size_t) plen + 1);
  if (h_prefix == NULL) return DX_E_NOMEM;
  memcpy(h_prefix,hd.prefix.data(),(size_t) plen + 1);
  DX_CUDA(ctx,cudaMemcpyAsync(d_prefix,h_prefix,(size_t) plen + 1,cudaMemcpyHostToDevice,ctx->stream));
  DX_CUDA(ctx,cudaMemsetAsync(d_flag,0,16,ctx->stream));
  int32_t *d_stat1 = d_flag + 1;                        // decode status of the final launch
  ph.mark("tables");

  QvTail *h_tail = (QvTail *) dx_hpin_get(ctx,sizeof(QvTail));
  if (h_tail == NULL) return DX_E_NOMEM;

  if (h_entry_off != NULL)
    { // ---- entry starts known -------------------------------------------------------------------
      const size_t N = (size_t) nentries;
      if (N == 0) { *out_len = 0; *handled = true; return DX_OK; }
      QvPlanArrays pa;
      int64_t *d_estart = (int64_t *) dx_arena_get(ctx,N*8);
      int64_t *d_wpre   = (int64_t *) dx_arena_get(ctx,(N+1)*8);
      int64_t *d_opre   = (int64_t *) dx_arena_get(ctx,(N+1)*8);
      uint32_t *d_len   = (uint32_t *) dx_arena_get(ctx,N*4);
      int32_t *d_well   = (int32_t *) dx_arena_get(ctx,N*4);
      QvDecEntry *d_ent = (QvDecEntry *) dx_arena_get(ctx,N*sizeof(QvDecEntry));
      if (!alloc_plan(ctx,N,pa) || !d_estart || !d_wpre || !d_opre || !d_len || !d_well || !d_ent) return DX_E_NOMEM;
      DX_CUDA(ctx,cudaMemcpyAsync(d_estart,h_entry_off,N*8,cudaMemcpyHostToDevice,ctx->stream));
      if ((rc = dxk_qv_known_prep(ctx,d_in,n,d_estart,(int64_t) N,pa,d_flag)) != DX_OK) return rc;
      if ((rc = dxk_scan_u32(ctx,pa.delta,(int64_t) N,d_wpre)) != DX_OK) return rc;
      if ((rc = dxk_qv_text_len(ctx,(int64_t) N,NULL,pa,d_wpre,NULL,well_in,plen,d_len,d_well,d_flag)) != DX_OK) return rc;
      if ((rc = dxk_scan_u32(ctx,d_len,(int64_t) N,d_opre)) != DX_OK) return rc;
      if ((rc = dxk_qv_build_ent(ctx,(int64_t) N,NULL,pa,d_well,d_opre,d_len,NULL,d_ent,NULL,NULL,NULL)) != DX_OK) return rc;
      if ((rc = make_tables()) != DX_OK) return rc;
      int32_t *h_rlen  = (int32_t *) dx_hpin_get(ctx,N*4);
      int32_t *h_order = (int32_t *) dx_hpin_get(ctx,N*4);
      int32_t *d_order = (int32_t *) dx_arena_get(ctx,N*4);
      int64_t *d_endat = (int64_t *) dx_arena_get(ctx,N*8);  // entry i ends where entry i+1 starts
      if (!h_rlen || !h_order || !d_order || !d_endat) return DX_E_NOMEM;
      const int64_t image_end = (int64_t) n;
      if (N > 1) DX_CUDA(ctx,cudaMemcpyAsync(d_endat,h_entry_off+1,(N-1)*8,cudaMemcpyHostToDevice,ctx->stream));
      DX_CUDA(ctx,cudaMemcpyAsync(d_endat+N-1,&image_end,8,cudaMemcpyHostToDevice,ctx->stream));
      DX_CUDA(ctx,cudaMemcpyAsync(h_rlen,pa.rlen,N*4,cudaMemcpyDeviceToHost,ctx->stream));
      DX_CUDA(ctx,cudaMemcpyAsync(&h_tail->total,d_opre+N,8,cudaMemcpyDeviceToHost,ctx->stream));
      DX_CUDA(ctx,cudaMemcpyAsync(&h_tail->flag,d_flag,4,cudaMemcpyDeviceToHost,ctx->stream));
      DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
      ph.mark("plan");
      if (h_tail->flag == 1) return dx_fail(ctx,DX_E_TRUNC,"compressed image ends inside an entry header");
      if (h_tail->flag == 2) return dx_fail(ctx,DX_E_FORMAT,"unusable read length in an entry header");
      if ((size_t) h_tail->total > cap)
        return dx_fail_cap(ctx,(size_t) (h_tail->total),cap);
      const int64_t n_coop = ticket_plan(ctx,h_rlen,N,h_order);
      DX_CUDA(ctx,cudaMemcpyAsync(d_order,h_order,N*4,cudaMemcpyHostToDevice,ctx->stream));
      if ((rc = dxk_qv_decode6x(ctx,d_in,n,d_tab4,coding.delchar,coding.subchar,upper,1,(int64_t) N,pa.fs,pa.rlen,
                                d_ent,d_prefix,plen,d_out,NULL,d_stat1,NULL,d_order,NULL,n_coop,d_endat)) != DX_OK) return rc;
      DX_CUDA(ctx,cudaMemcpyAsync(&h_tail->flag,d_stat1,4,cudaMemcpyDeviceToHost,ctx->stream));
      DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
      ph.mark("decode");
      ph.report("undexqv (index known)");
      if (h_tail->flag) return dx_fail(ctx,DX_E_TRUNC,"Could not read more bits (Decode)");
      if (ctx->keep_index)
        { std::vector<QvDecEntry> he; std::vector<int64_t> hfs;
          if ((rc = download(ctx,d_ent,N,he)) != DX_OK) return rc;
          if ((rc = download(ctx,pa.fs,N,hfs)) != DX_OK) return rc;
          std::vector<int64_t> end_off(h_entry_off + 1,h_entry_off + N);
          end_off.push_back((int64_t) n);
          set_last_index(ctx,N,he.data(),hfs.data(),end_off.data());
        }
      *out_len = (size_t) h_tail->total;
      *handled = true;
      return DX_OK;
    }

  // ---- entry starts unknown: candidates, speculative decode, verified chain --------------------------
  int64_t *d_q = NULL, nc = 0;
  ctx->overlap_arg = &deferred;
  ctx->overlap_fn = [](void *p) { Deferred *d = (Deferred *) p; d->rc = (*d->fn)(); };
  rc = dxk_index_positions(ctx,DX_PRED_QVCAND,d_in,n,first + 1,&d_q,&nc);
  if (ctx->overlap_fn != NULL)                          // the index took a route without the hook
    { ctx->overlap_fn = NULL;
      deferred.rc = make_tables();
    }
  if (rc != DX_OK) return rc;
  if (deferred.rc != DX_OK) return deferred.rc;
  ph.mark("index");
  const size_t N = (size_t) nc;
  if (N == 0) return DX_OK;                             // empty or all entries missed: general path
  QvCands c;
  if ((rc = qv_cands_prep(ctx,d_in,n,first,d_q,nc,qv_minbits(coding),h_tail,c)) != DX_OK) return rc;
  // The layout of the text IF the entries are exactly the candidates k_qv_direct_prep keeps (not within
  // 13 bytes of a later one, fields in the range of real headers) and every well delta but the first is below 255
  // (no 0xff delta bytes; true of real data, where consecutive wells are a few holes apart): wells and text
  // offsets are then prefix sums over the candidates, and the decoder can write headers and lines
  // straight into place.  The chain below still decides; when it disagrees the lines are decoded
  // again into a scratch image and moved (k_qv_assemble), as if nothing had been assumed.
  int64_t *d_wpre = (int64_t *) dx_arena_get(ctx,(N+1)*8);
  int64_t *d_opre = (int64_t *) dx_arena_get(ctx,(N+1)*8);
  uint32_t *d_len = (uint32_t *) dx_arena_get(ctx,N*4 + 4);
  int32_t *d_well = (int32_t *) dx_arena_get(ctx,N*4 + 4);
  QvDecEntry *d_ent = (QvDecEntry *) dx_arena_get(ctx,(N+1)*sizeof(QvDecEntry));
  int32_t *d_rlen_d = (int32_t *) dx_arena_get(ctx,N*4 + 4);   // rlen, -1 for candidates outside that layout
  int32_t *d_flag2 = d_flag + 2;                        // unusable length in some candidate
  uint8_t *d_keep = (uint8_t *) dx_arena_get(ctx,N + 4);         // 1: part of that layout
  if (!d_wpre || !d_opre || !d_len || !d_well || !d_ent || !d_rlen_d || !d_keep) return DX_E_NOMEM;
  if ((rc = dxk_qv_direct_prep(ctx,d_q,nc,c.pa,d_rlen_d,d_keep)) != DX_OK) return rc;
  if ((rc = dxk_scan_u32(ctx,c.pa.delta,nc,d_wpre)) != DX_OK) return rc;
  if ((rc = dxk_qv_text_len(ctx,nc,NULL,c.pa,d_wpre,NULL,well_in,plen,d_len,d_well,d_flag2,d_rlen_d)) != DX_OK) return rc;
  if ((rc = dxk_scan_u32(ctx,d_len,nc,d_opre)) != DX_OK) return rc;
  if ((rc = dxk_qv_build_ent(ctx,nc,NULL,c.pa,d_well,d_opre,d_len,NULL,d_ent,NULL,NULL,NULL)) != DX_OK) return rc;
  int64_t *h_tot  = (int64_t *) dx_hpin_get(ctx,16);
  uint8_t *h_keep = (uint8_t *) dx_hpin_get(ctx,N);
  if (!h_tot || !h_keep) return DX_E_NOMEM;
  DX_CUDA(ctx,cudaMemcpyAsync(h_keep,d_keep,N,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaMemcpyAsync(h_tot,d_opre+N,8,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaMemcpyAsync(&h_tail->flag,d_flag2,4,cudaMemcpyDeviceToHost,ctx->stream));
  if ((rc = qv_cands_plan(ctx,c,false)) != DX_OK) return rc;
  ph.mark("prep");
  const int64_t direct_total = h_tot[0];
  bool direct = !ctx->route[DXR_NO_DIRECT] && c.n_coop == (int64_t) N && h_tail->flag == 0 &&
                direct_total >= 0 && (size_t) direct_total <= cap;
  if (direct)
    rc = dxk_qv_decode6x(ctx,d_in,n,d_tab4,coding.delchar,coding.subchar,upper,3,nc,c.pa.fs,d_rlen_d,d_ent,d_prefix,plen,
                         d_out,c.d_soff,c.d_stat,c.d_limit,c.d_order,NULL,c.n_coop);
  else
    rc = qv_cands_decode(ctx,d_in,n,d_tab4,coding,upper,c);
  if (rc != DX_OK) return rc;
  if (direct && !ctx->keep_index)
    { // the usual end of the call: the device checks that the decode confirmed the layout (the chain
      // walk below as a predicate over independent candidates); the host reads two words
      int32_t *d_chk = (int32_t *) dx_arena_get(ctx,8);
      int32_t *h_chk = (int32_t *) dx_hpin_get(ctx,8);
      if (!d_chk || !h_chk) return DX_E_NOMEM;
      DX_CUDA(ctx,cudaMemsetAsync(d_chk,0,8,ctx->stream));
      if ((rc = dxk_qv_chain_check(ctx,d_q,nc,d_keep,d_rlen_d,c.d_stat,c.d_soff,c.d_last,c.d_ffrun,first,n,d_chk)) != DX_OK)
        return rc;
      DX_CUDA(ctx,cudaMemcpyAsync(h_chk,d_chk,8,cudaMemcpyDeviceToHost,ctx->stream));
      DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
      ph.mark("decode");
      if (h_chk[0] == 0 && h_chk[1] > 0)             // (no kept candidate at all proves nothing)
        { if (ctx->route[DXR_DEBUG])
            fprintf(stderr,"[dexb200 debug] undexqv: %zu candidates, %d entries, decoded in place (checked on the device)\n",
                    N,h_chk[1]);
          ph.report("undexqv (entries discovered)");
          *out_len = (size_t) direct_total;
          *handled = true;
          return DX_OK;
        }
    }
  DX_CUDA(ctx,cudaMemcpyAsync(c.h_soff,c.d_soff,N*48,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaMemcpyAsync(c.h_stat,c.d_stat,N*4,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  ph.mark("decode");

  // the chain (dx_chain.h) over the whole image
  const DxChainIn ci = { c.h_q, c.h_ffrun, c.h_last, c.h_stat, c.h_soff, h_keep, (int64_t) N, (int64_t) first, (int64_t) n };
  int64_t m = 0;
  bool as_assumed = true;                 // the entries are the candidates of the assumed layout, with its deltas
  if (!dx_chain_walk(ci,well_in,c.h_cand,c.h_well,&m,&as_assumed)) return DX_OK;          // general path
  const size_t M = (size_t) m;
  ph.mark("chain");
  size_t total = (size_t) direct_total;
  if (direct && as_assumed)
    { if (ctx->route[DXR_DEBUG])
        fprintf(stderr,"[dexb200 debug] undexqv: %zu candidates, %zu entries, decoded in place\n",N,M);
    }
  else
    { if (direct)
        { // the assumption did not hold: the same candidates once more, lines only, into the scratch image
          // (soff / status do not depend on where the text goes)
          if (ctx->route[DXR_DEBUG])
            fprintf(stderr,"[dexb200 debug] undexqv: %zu candidates (%zu in the assumed layout), %zu entries: "
                           "not as assumed, decoding again\n",N,N - (size_t) std::count(h_keep,h_keep + N,0),M);
          if ((rc = qv_cands_decode(ctx,d_in,n,d_tab4,coding,upper,c)) != DX_OK) return rc;
          direct = false;
        }
      if ((rc = qv_layout(ctx,c,M,plen,d_flag,false,&total)) != DX_OK) return rc;
      if (total > cap) return dx_fail_cap(ctx,total,cap);
      if ((rc = dxk_qv_assemble(ctx,c.d_tmp,c.tmp_n,c.d_ent,c.d_src,(int64_t) M,d_prefix,plen,d_out)) != DX_OK) return rc;
      DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
      ph.mark("assemble");
    }
  ph.report("undexqv (entries discovered)");
  if (ctx->keep_index)
    { std::vector<QvDecEntry> he;
      if ((rc = download(ctx,direct ? d_ent : c.d_ent,direct ? N : M,he)) != DX_OK) return rc;   // direct: one row per candidate
      std::vector<QvDecEntry> ent(M);
      std::vector<int64_t> stream_off(M), end_off(M);
      for (size_t i = 0; i < M; i++)
        { const size_t k = (size_t) c.h_cand[i];
          ent[i] = he[direct ? k : i]; stream_off[i] = c.h_q[k] + 12; end_off[i] = c.h_soff[6*k + 5];
        }
      set_last_index(ctx,M,ent.data(),stream_off.data(),end_off.data());
    }
  *out_len = total;
  *handled = true;
  return DX_OK;
}

extern "C" int dx_undexqv_dev(dx_ctx *ctx, const uint8_t *d_in, size_t n, int upper,
                              uint8_t *d_out, size_t cap, size_t *out_len,
                              const int64_t *h_entry_off, int64_t nentries, int32_t well_in)
{ if (ctx == NULL || out_len == NULL) return DX_E_ARG;
  int rc;
  *out_len = 0;
  if ((rc = check_buf(ctx,d_in,"image")) != DX_OK) return rc;
  cudaSetDevice(ctx->device);
  dx_arena_reset(ctx);
  { bool handled = false;
    if (d_out != NULL && (rc = undexqv_fast(ctx,d_in,n,upper,d_out,cap,out_len,h_entry_off,nentries,well_in,
                                            &handled)) != DX_OK) return rc;
    if (handled) return DX_OK;
    dx_arena_reset(ctx);
  }
  if (ctx->last_index) ((std::vector<dx_index_row> *) ctx->last_index)->clear();
  QvPlan plan;
  if ((rc = plan_undexqv(ctx,d_in,n,h_entry_off,nentries,well_in,true,upper,plan)) != DX_OK) return rc;
  if (plan.text_len > cap)
    return dx_fail_cap(ctx,(size_t) (plan.text_len),cap);
  const size_t N = plan.ent.size();
  QvDecEntry *d_ent = (QvDecEntry *) dx_arena_get(ctx,N*sizeof(QvDecEntry));
  int32_t *d_stat = (int32_t *) dx_arena_get(ctx,4);
  if (!d_ent || !d_stat) return DX_E_NOMEM;
  if ((rc = upload(ctx,d_ent,plan.ent.data(),N)) != DX_OK) return rc;
  DX_CUDA(ctx,cudaMemsetAsync(d_stat,0,4,ctx->stream));
  const dx_qv_coding &cd = plan.coding;
  if (plan.spec)
    { // the lines are already decoded (scratch image): write the headers and move them into place;
      // entries the candidate filter missed (rare) are decoded now
      int64_t *d_src = (int64_t *) dx_arena_get(ctx,N*8);
      if (!d_src) return DX_E_NOMEM;
      if ((rc = upload(ctx,d_src,plan.src.data(),N)) != DX_OK) return rc;
      if ((rc = dxk_qv_assemble(ctx,plan.d_tmp,plan.tmp_n,d_ent,d_src,(int64_t) N,plan.d_prefix,plan.plen,
                                d_out)) != DX_OK) return rc;
      std::vector<size_t> miss;
      for (size_t i = 0; i < N; i++) if (plan.src[i] < 0) miss.push_back(i);
      rc = DX_OK;
      if (!miss.empty())
        { const size_t K = miss.size();
          std::vector<int64_t> st, stall;
          std::vector<int32_t> rl, rlall;
          if ((rc = download(ctx,plan.d_start,N,stall)) != DX_OK) return rc;
          if ((rc = download(ctx,plan.d_rlen,N,rlall)) != DX_OK) return rc;
          std::vector<QvDecEntry> me(K);
          st.resize(K); rl.resize(K);
          for (size_t k = 0; k < K; k++) { st[k] = stall[miss[k]]; rl[k] = rlall[miss[k]]; me[k] = plan.ent[miss[k]]; }
          int64_t *d_st = (int64_t *) dx_arena_get(ctx,K*8);
          int32_t *d_rl = (int32_t *) dx_arena_get(ctx,K*4);
          QvDecEntry *d_me = (QvDecEntry *) dx_arena_get(ctx,K*sizeof(QvDecEntry));
          if (!d_st || !d_rl || !d_me) return DX_E_NOMEM;
          if ((rc = upload(ctx,d_st,st.data(),K)) != DX_OK) return rc;
          if ((rc = upload(ctx,d_rl,rl.data(),K)) != DX_OK) return rc;
          if ((rc = upload(ctx,d_me,me.data(),K)) != DX_OK) return rc;
          rc = dxk_qv_decode5(ctx,d_in,n,plan.d_tab4,cd.delchar,cd.subchar,upper,1,(int64_t) K,d_st,d_rl,d_me,
                              plan.d_prefix,plan.plen,d_out,NULL,d_stat);
        }
    }
  else if (plan.v2)
    { int64_t *d_endat = NULL;                                 // known offsets: entry i ends where i+1 starts
      if (h_entry_off != NULL && plan.ix_end.size() == N)
        { if ((d_endat = (int64_t *) dx_arena_get(ctx,N*8)) == NULL) return DX_E_NOMEM;
          if ((rc = upload(ctx,d_endat,plan.ix_end.data(),N)) != DX_OK) return rc;
        }
      rc = dxk_qv_decode5x(ctx,d_in,n,plan.d_tab4,cd.delchar,cd.subchar,upper,1,(int64_t) N,
                           plan.d_start,plan.d_rlen,d_ent,plan.d_prefix,plan.plen,d_out,NULL,d_stat,
                           NULL,NULL,NULL,d_endat);
    }
  else
    rc = dxk_qv_decode(ctx,d_in,n,plan.d_tab,cd.delchar,cd.subchar,cd.flip,upper,d_ent,plan.d_soff,
                       (int64_t) N,plan.d_prefix,plan.plen,d_out,d_stat);
  if (rc != DX_OK) return rc;
  int32_t stat = 0;
  DX_CUDA(ctx,cudaMemcpyAsync(&stat,d_stat,4,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  if (stat) return dx_fail(ctx,DX_E_TRUNC,"Could not read more bits (Decode)");
  if (ctx->keep_index && ctx->last_index && plan.ix_fs.size() == N)
    set_last_index(ctx,N,plan.ent.data(),plan.ix_fs.data(),plan.ix_end.data());
  *out_len = plan.text_len;
  return DX_OK;
}

// Batched Load_QVentry (DB.c:2575-2621): the streams of entry i start at d_in[h_stream_off[i]] and
// hold h_rlen[i] positions; its five lines, each followed by a newline, go to
// d_out[off[i] .. off[i] + 5*(rlen+1)) with off = exclusive prefix sum (returned in h_out_off).
extern "C" int dx_qv_load_entries_dev(dx_ctx *ctx, const uint8_t *d_in, size_t n, const dx_qv_coding *coding,
                                      const int64_t *h_stream_off, const int32_t *h_rlen, int64_t nentries,
                                      int upper, uint8_t *d_out, size_t cap, int64_t *h_out_off,
                                      int64_t *h_end_off)
{ if (ctx == NULL || coding == NULL || nentries < 0 || (nentries > 0 && (!h_stream_off || !h_rlen))) return DX_E_ARG;
  int rc;
  if ((rc = check_buf(ctx,d_in,"image")) != DX_OK) return rc;
  if (coding->flip) return dx_fail(ctx,DX_E_KEY,"dx_qv_load_entries_dev: foreign-endian codings are not supported");
  cudaSetDevice(ctx->device);
  dx_arena_reset(ctx);
  const size_t N = (size_t) nentries;
  std::vector<int64_t> toff(N + 1,0);
  for (size_t i = 0; i < N; i++)
    { if (h_rlen[i] < 0 || h_rlen[i] >= (1 << 24) || h_stream_off[i] < 0 || (size_t) h_stream_off[i] > n)
        return dx_fail(ctx,DX_E_ARG,"dx_qv_load_entries_dev: entry %zu out of range",i);
      toff[i+1] = toff[i] + 5*((int64_t) h_rlen[i] + 1);
    }
  if (h_out_off) memcpy(h_out_off,toff.data(),(N + 1)*8);
  if (N == 0) return DX_OK;
  if ((size_t) toff[N] > cap)
    return dx_fail_cap(ctx,(size_t) (toff[N]),cap);
  QvDecTables4 *d_tab4 = (QvDecTables4 *) dx_arena_get(ctx,sizeof(QvDecTables4));
  if (d_tab4 == NULL) return DX_E_NOMEM;
  if ((rc = qv_tables4(ctx,coding,NULL,false,d_tab4)) != DX_OK) return rc;
  int64_t *d_start = (int64_t *) dx_arena_get(ctx,N*8);
  int32_t *d_rlen  = (int32_t *) dx_arena_get(ctx,N*4);
  int64_t *d_toff  = (int64_t *) dx_arena_get(ctx,(N+1)*8);
  int64_t *d_soff  = (int64_t *) dx_arena_get(ctx,N*48);
  int32_t *d_stat  = (int32_t *) dx_arena_get(ctx,N*4);
  int32_t *d_order = (int32_t *) dx_arena_get(ctx,N*4);
  if (!d_start || !d_rlen || !d_toff || !d_soff || !d_stat || !d_order) return DX_E_NOMEM;
  std::vector<int32_t> order(N);
  const int64_t n_coop = ticket_plan(ctx,h_rlen,N,order.data());
  if ((rc = upload(ctx,d_start,h_stream_off,N)) != DX_OK) return rc;
  if ((rc = upload(ctx,d_rlen,h_rlen,N)) != DX_OK) return rc;
  if ((rc = upload(ctx,d_toff,toff.data(),N + 1)) != DX_OK) return rc;
  if ((rc = upload(ctx,d_order,order.data(),N)) != DX_OK) return rc;
  if ((rc = dxk_qv_decode6x(ctx,d_in,n,d_tab4,coding->delchar,coding->subchar,upper,2,(int64_t) N,d_start,d_rlen,
                            NULL,NULL,0,d_out,d_soff,d_stat,NULL,d_order,d_toff,n_coop)) != DX_OK) return rc;
  std::vector<int32_t> stat;
  if ((rc = download(ctx,d_stat,N,stat)) != DX_OK) return rc;
  for (size_t i = 0; i < N; i++)
    if (stat[i]) return dx_fail(ctx,DX_E_TRUNC,"Could not read more bits (Decode), entry %zu",i + 1);
  if (h_end_off != NULL)
    { std::vector<int64_t> so;
      if ((rc = download(ctx,d_soff,N*6,so)) != DX_OK) return rc;
      for (size_t i = 0; i < N; i++) h_end_off[i] = so[6*i + 5];
    }
  return DX_OK;
}

extern "C" int dx_undexqv_size_dev(dx_ctx *ctx, const uint8_t *d_in, size_t n, size_t *out_len)
{ if (ctx == NULL || out_len == NULL) return DX_E_ARG;
  int rc;
  *out_len = 0;
  if ((rc = check_buf(ctx,d_in,"image")) != DX_OK) return rc;
  cudaSetDevice(ctx->device);
  dx_arena_reset(ctx);
  QvPlan plan;
  if ((rc = plan_undexqv(ctx,d_in,n,NULL,0,0,false,0,plan)) != DX_OK) return rc;
  *out_len = plan.text_len;
  return DX_OK;
}

// ================================================================================================
//  *_host entry points: stage through device memory, copies included
// ================================================================================================

static int stage_in(dx_ctx *ctx, const uint8_t *h, size_t n)
{ int rc;
  cudaSetDevice(ctx->device);
  if ((rc = ensure_io(ctx,&ctx->io_in,&ctx->io_in_cap,n)) != DX_OK) return rc;
  if (n > 0)
    DX_CUDA(ctx,cudaMemcpyAsync(ctx->io_in,h,n,cudaMemcpyHostToDevice,ctx->stream));
  return DX_OK;
}

static int stage_out(dx_ctx *ctx, uint8_t *h, size_t n)
{ if (n > 0)
    DX_CUDA(ctx,cudaMemcpyAsync(h,ctx->io_out,n,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  return DX_OK;
}

extern "C" int dx_dexta_host(dx_ctx *ctx, int kind, const uint8_t *h_text, size_t n,
                             uint8_t *h_out, size_t cap, size_t *out_len)
{ if (ctx == NULL || h_text == NULL || h_out == NULL || out_len == NULL) return DX_E_ARG;
  int rc;
  if ((rc = stage_in(ctx,h_text,n)) != DX_OK) return rc;
  if ((rc = ensure_io(ctx,&ctx->io_out,&ctx->io_out_cap,cap)) != DX_OK) return rc;
  if ((rc = dx_dexta_dev(ctx,kind,ctx->io_in,n,ctx->io_out,cap,out_len)) != DX_OK) return rc;
  return stage_out(ctx,h_out,*out_len);
}

extern "C" int dx_undexta_size_host(dx_ctx *ctx, int kind, const uint8_t *h_in, size_t n, int width,
                                    size_t *out_len)
{ if (ctx == NULL || h_in == NULL || out_len == NULL) return DX_E_ARG;
  int rc;
  if ((rc = stage_in(ctx,h_in,n)) != DX_OK) return rc;
  return dx_undexta_size_dev(ctx,kind,ctx->io_in,n,width,out_len);
}

extern "C" int dx_undexta_host(dx_ctx *ctx, int kind, const uint8_t *h_in, size_t n, int width,
                               int upper, uint8_t *h_out, size_t cap, size_t *out_len)
{ if (ctx == NULL || h_in == NULL || h_out == NULL || out_len == NULL) return DX_E_ARG;
  int rc;
  if ((rc = stage_in(ctx,h_in,n)) != DX_OK) return rc;
  if ((rc = ensure_io(ctx,&ctx->io_out,&ctx->io_out_cap,cap)) != DX_OK) return rc;
  if ((rc = dx_undexta_dev(ctx,kind,ctx->io_in,n,width,upper,ctx->io_out,cap,out_len)) != DX_OK) return rc;
  return stage_out(ctx,h_out,*out_len);
}

extern "C" int dx_dexqv_host(dx_ctx *ctx, const uint8_t *h_text, size_t n, int lossy,
                             uint8_t *h_out, size_t cap, size_t *out_len)
{ if (ctx == NULL || h_text == NULL || h_out == NULL || out_len == NULL) return DX_E_ARG;
  int rc;
  if ((rc = stage_in(ctx,h_text,n)) != DX_OK) return rc;
  if ((rc = ensure_io(ctx,&ctx->io_out,&ctx->io_out_cap,cap)) != DX_OK) return rc;
  if ((rc = dx_dexqv_dev(ctx,ctx->io_in,n,lossy,ctx->io_out,cap,out_len)) != DX_OK) return rc;
  return stage_out(ctx,h_out,*out_len);
}

// ------------------------------------------------------------------------------------------------
//  One byte range of a .dexqv image: the entries whose FIRST byte (the first well-delta byte,
//  undexqv.c:119-208 reads the delta first) lies in [a, b).  Three steps, so that callers with one
//  range per GPU run the expensive one everywhere at once and hand on only the chain's position:
//    qv_range_decode  the range's candidates, decoded speculatively (qv_cands_prep / plan / decode);
//    qv_range_chain   the host walk from the carried position and well, bounded to the range
//                     (dx_chain_walk_general: an entry the candidates miss is read and decoded by
//                     itself, as plan_undexqv's general path does);
//    qv_range_text    the text of the chain (qv_layout + k_qv_assemble); after a walk that needed the
//                     slow path, the chain's entries are decoded once more as the only candidates.
//  The kernels see the image bytes [base, base + w_n) at w_in, base at most 4096 bytes in front of
//  the range (as far back as they look) and 16-byte aligned.  undexqv_pipe runs its windows through
//  these steps; dx_undexqv_range_* expose them.
// ------------------------------------------------------------------------------------------------
struct QvRange
{ dx_qv_coding  coding;             // set-up, the same for every range of one image
  int           plen, minbits, upper;
  int64_t       first;              // first byte behind the coding header
  QvDecTables4 *d_tab4;
  char         *d_prefix;
  int32_t      *d_flag;
  QvTail       *h_tail;
  bool          by_kernel;          // small transfers through dxk_fetch (qv_copy)
  const uint8_t *w_in;              // the range
  size_t        w_n;
  int64_t       base, a, b;
  QvCands       c;
  std::vector<DxChainEntry> ent;    // the chain, in window coordinates
  bool          slow;               // some entry of it is no candidate of c
};

static void qv_range_free(dx_ctx *ctx)
{ delete (QvRange *) ctx->qv_range;
  ctx->qv_range = NULL;
}

static int qv_range_setup(dx_ctx *ctx, const QvHead &hd, int upper, bool by_kernel, QvRange &R)
{ R.coding = hd.coding; R.plen = hd.plen; R.first = (int64_t) hd.first; R.upper = upper;
  R.by_kernel = by_kernel; R.minbits = qv_minbits(hd.coding);
  QvDecTables4 *h4 = (QvDecTables4 *) dx_hpin_get(ctx,sizeof(QvDecTables4));
  char *h_prefix = (char *) dx_hpin_get(ctx,(size_t) R.plen + 1);
  R.d_tab4   = (QvDecTables4 *) dx_arena_get(ctx,sizeof(QvDecTables4));
  R.d_prefix = (char *) dx_arena_get(ctx,(size_t) R.plen + 1);
  R.d_flag   = (int32_t *) dx_arena_get(ctx,16);
  R.h_tail   = (QvTail *) dx_hpin_get(ctx,sizeof(QvTail));
  if (!h4 || !h_prefix || !R.d_tab4 || !R.d_prefix || !R.d_flag || !R.h_tail) return DX_E_NOMEM;
  int rc;
  if ((rc = qv_tables4(ctx,&hd.coding,h4,by_kernel,R.d_tab4)) != DX_OK) return rc;
  memcpy(h_prefix,hd.prefix.data(),(size_t) R.plen + 1);
  if ((rc = qv_copy(ctx,by_kernel,R.d_prefix,h_prefix,(size_t) R.plen + 1)) != DX_OK) return rc;
  DX_CUDA(ctx,cudaMemsetAsync(R.d_flag,0,16,ctx->stream));
  return DX_OK;
}

// the window origin of a range whose entries start at a >= first, in a buffer starting at image offset buf_off
static int64_t qv_range_base(int64_t a, int64_t buf_off)
{ const int64_t lo = (a > 4096) ? a - 4096 : 0;
  return buf_off + ((lo - buf_off) & ~(int64_t) 15);
}

static int qv_range_decode(dx_ctx *ctx, QvRange &R, const uint8_t *w_in, size_t w_n, int64_t base, int64_t a, int64_t b)
{ R.w_in = w_in; R.w_n = w_n; R.base = base; R.a = a; R.b = b;
  R.c = QvCands();
  R.ent.clear(); R.slow = false;
  if (b <= a) return DX_OK;
  const int64_t wfirst = a - base;
  const int64_t scan_end = (b + 64 < base + (int64_t) w_n) ? b + 64 : base + (int64_t) w_n;
  int64_t *d_q = NULL, nc = 0;
  int rc;
  if ((rc = dxk_index_positions(ctx,DX_PRED_QVCAND,w_in,(size_t) (scan_end - base),(size_t) wfirst + 1,&d_q,&nc)) != DX_OK)
    return rc;
  if (nc == 0) return DX_OK;
  if ((rc = qv_cands_prep(ctx,w_in,w_n,(size_t) wfirst,d_q,nc,R.minbits,R.h_tail,R.c)) != DX_OK ||
      (rc = qv_cands_plan(ctx,R.c,R.by_kernel)) != DX_OK ||
      (rc = qv_cands_decode(ctx,w_in,w_n,R.d_tab4,R.coding,R.upper,R.c)) != DX_OK ||
      (rc = qv_copy(ctx,R.by_kernel,R.c.h_soff,R.c.d_soff,R.c.N*48)) != DX_OK ||
      (rc = qv_copy(ctx,R.by_kernel,R.c.h_stat,R.c.d_stat,R.c.N*4)) != DX_OK) return rc;
  return DX_OK;
}

// Bytes an entry of rlen positions takes behind its fields, at most: in a run-length coded stream every
// position a run code and a symbol code, both escaped; two bits per tag; each stream padded to words.
static int64_t qv_entry_bound(const dx_qv_coding &cd, int64_t rlen)
{ auto maxlen = [&](int k) { int m = 0; for (int x = 0; x < 256; x++) m = std::max(m,(int) cd.tab[k].lens[x]); return (int64_t) m; };
  const int64_t bits[4] = { maxlen(0) + 8 + (cd.delchar >= 0 ? maxlen(1) + 16 : 0), maxlen(2) + 8, maxlen(3) + 8,
                            maxlen(4) + 8 + (cd.subchar >= 0 ? maxlen(5) + 16 : 0) };
  int64_t bytes = (rlen + 3) / 4 + 8;
  for (int s = 0; s < 4; s++) bytes += (rlen * bits[s] + 7) / 8 + 8;
  return bytes;
}

// DX_E_CAP: the range's buffer ends before the entry at image offset `at` does; it needs the image up to `need`
static int qv_range_short(dx_ctx *ctx, const QvRange &R, int64_t at, int64_t need)
{ dx_fail(ctx,DX_E_CAP,"the entry at image offset %lld runs past the end of the buffer (%lld): it needs the image up to %lld",
          (long long) at,(long long) (R.base + (int64_t) R.w_n),(long long) need);
  ctx->need_bytes = (size_t) need;
  return DX_E_CAP;
}

struct QvSlowUser { dx_ctx *ctx; QvRange *R; };

// dx_chain_walk_general's slow path: the entry at cur (window coordinates) read and decoded by itself
static int qv_range_slow(void *user, int64_t cur, int64_t *q, int64_t *end, int32_t *delta)
{ dx_ctx *ctx = ((QvSlowUser *) user)->ctx;
  const QvRange &R = *((QvSlowUser *) user)->R;
  const int64_t n = (int64_t) R.w_n;
  std::vector<uint8_t> win;
  int64_t p = cur;
  int32_t add = 0;
  int rc;
  for (;;)                                                  // the delta bytes: 0xff ... 0xff, d
    { if ((rc = peek(ctx,R.w_in,R.w_n,(size_t) p,4096,win)) != DX_OK) return rc;
      size_t k = 0;
      while (k < win.size() && win[k] == 0xff) k++;
      add += 255 * (int32_t) k; p += (int64_t) k;
      if (k < win.size()) { add += win[k]; p += 1; break; }
      if (p >= n)                                           // a delta is at most 2^31 wells: 8 421 505 bytes
        return qv_range_short(ctx,R,R.base + cur,R.base + cur + 8421505 + 12);
    }
  if ((rc = peek(ctx,R.w_in,R.w_n,(size_t) p,12,win)) != DX_OK) return rc;
  if (win.size() < 12) return qv_range_short(ctx,R,R.base + cur,R.base + p + 12 + 65536);
  const int32_t rlen = le32(win.data() + 4) - le32(win.data());
  if (rlen < 0 || rlen >= (1 << 24))
    return dx_fail(ctx,DX_E_FORMAT,"unusable read length %d in the entry header at image offset %lld",rlen,
                   (long long) (R.base + p));
  int64_t *d_start = (int64_t *) dx_arena_get(ctx,8);
  int32_t *d_rlen  = (int32_t *) dx_arena_get(ctx,4);
  int64_t *d_soff  = (int64_t *) dx_arena_get(ctx,48);
  int32_t *d_stat  = (int32_t *) dx_arena_get(ctx,4);
  if (!d_start || !d_rlen || !d_soff || !d_stat) return DX_E_NOMEM;
  const int64_t start = p + 12;
  if ((rc = upload(ctx,d_start,&start,1)) != DX_OK || (rc = upload(ctx,d_rlen,&rlen,1)) != DX_OK) return rc;
  if ((rc = dxk_qv_decode5(ctx,R.w_in,R.w_n,R.d_tab4,R.coding.delchar,R.coding.subchar,0,0,1,d_start,d_rlen,
                           NULL,NULL,0,NULL,d_soff,d_stat)) != DX_OK) return rc;
  std::vector<int64_t> so; std::vector<int32_t> st;
  if ((rc = download(ctx,d_soff,6,so)) != DX_OK || (rc = download(ctx,d_stat,1,st)) != DX_OK) return rc;
  if (st[0] != 0 || so[5] > n || so[5] <= cur)
    { const int64_t need = R.base + start + qv_entry_bound(R.coding,rlen);
      if (need > R.base + n) return qv_range_short(ctx,R,R.base + cur,need);
      return dx_fail(ctx,DX_E_TRUNC,"Could not read more bits (Decode), entry at image offset %lld",(long long) (R.base + cur));
    }
  *q = p; *end = so[5]; *delta = add;
  return DX_OK;
}

static int qv_range_chain(dx_ctx *ctx, QvRange &R, int64_t cur_in, int32_t well_in, int64_t *cur_out, int32_t *well_out)
{ DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));          // the candidates' ends and status
  const QvCands &c = R.c;
  const DxChainIn ci = { c.h_q, c.h_ffrun, c.h_last, c.h_stat, c.h_soff, NULL, (int64_t) c.N, R.a - R.base,
                         (int64_t) R.w_n, cur_in - R.base, R.b - R.base };
  QvSlowUser u = { ctx, &R };
  int64_t stop = 0;
  const int rc = dx_chain_walk_general(ci,well_in,qv_range_slow,&u,R.ent,&stop);
  if (rc != DX_OK) { R.ent.clear(); return rc; }
  R.slow = false;
  for (const DxChainEntry &e : R.ent) R.slow = R.slow || (e.cand < 0);
  *cur_out = stop + R.base;
  *well_out = R.ent.empty() ? well_in : R.ent.back().well;
  if (ctx->route[DXR_DEBUG] && R.slow)
    fprintf(stderr,"[dexb200 debug] undexqv range [%lld, %lld): %zu entries, some found by the slow path\n",
            (long long) R.a,(long long) R.b,R.ent.size());
  return DX_OK;
}

static int qv_range_text(dx_ctx *ctx, QvRange &R, uint8_t *d_out, size_t cap, size_t *out_len)
{ const size_t M = R.ent.size();
  *out_len = 0;
  if (M == 0) return DX_OK;
  int rc;
  bool redo = false;
  if (R.slow)
    { // entries the candidates did not give: the chain's own entries, decoded as the only candidates and
      // without the speculative decode's limit (which also gives up on entries that synchronise late)
      int64_t *h_q = (int64_t *) dx_hpin_get(ctx,M*8);
      int64_t *d_q = (int64_t *) dx_arena_get(ctx,M*8);
      if (!h_q || !d_q) return DX_E_NOMEM;
      for (size_t m = 0; m < M; m++) { h_q[m] = R.ent[m].q; R.ent[m].cand = (int32_t) m; }
      R.c = QvCands();
      QvCands &c = R.c;
      if ((rc = qv_copy(ctx,R.by_kernel,d_q,h_q,M*8)) != DX_OK ||
          (rc = qv_cands_prep(ctx,R.w_in,R.w_n,(size_t) (R.a - R.base),d_q,(int64_t) M,0,R.h_tail,c)) != DX_OK ||
          (rc = qv_cands_plan(ctx,c,R.by_kernel)) != DX_OK) return rc;
      if ((c.d_tmp = (uint8_t *) dx_arena_get(ctx,c.tmp_n + 64)) == NULL) return DX_E_NOMEM;
      if ((rc = dxk_qv_decode6x(ctx,R.w_in,R.w_n,R.d_tab4,R.coding.delchar,R.coding.subchar,R.upper,2,(int64_t) M,c.pa.fs,
                                c.pa.rlen,NULL,NULL,0,c.d_tmp,c.d_soff,c.d_stat,NULL,c.d_order,c.d_toff,c.n_coop)) != DX_OK ||
          (rc = qv_copy(ctx,R.by_kernel,c.h_stat,c.d_stat,M*4)) != DX_OK) return rc;
      R.slow = false;
      redo = true;
    }
  for (size_t m = 0; m < M; m++) { R.c.h_cand[m] = R.ent[m].cand; R.c.h_well[m] = R.ent[m].well; }
  size_t total = 0;
  if ((rc = qv_layout(ctx,R.c,M,R.plen,R.d_flag,R.by_kernel,&total)) != DX_OK) return rc;
  for (size_t m = 0; redo && m < M; m++)                     // (qv_layout waited for the stream)
    if (R.c.h_stat[m] != 0)
      return dx_fail(ctx,DX_E_TRUNC,"Could not read more bits (Decode), entry at image offset %lld",
                     (long long) (R.base + R.ent[m].q));
  if (total > cap) return dx_fail_cap(ctx,total,cap);
  if ((rc = dxk_qv_assemble(ctx,R.c.d_tmp,R.c.tmp_n,R.c.d_ent,R.c.d_src,(int64_t) M,R.d_prefix,R.plen,d_out)) != DX_OK)
    return rc;
  *out_len = total;
  return DX_OK;
}

extern "C" int dx_undexqv_range_dev(dx_ctx *ctx, const uint8_t *h_head, size_t head_n, const uint8_t *d_buf,
                                    size_t buf_n, int64_t buf_off, int64_t a, int64_t b, int upper, int64_t *first)
{ if (ctx == NULL) return DX_E_ARG;
  int rc;
  if (h_head == NULL) return dx_fail(ctx,DX_E_ARG,"dx_undexqv_range_dev: h_head is NULL");
  if ((rc = check_buf(ctx,d_buf,"range buffer")) != DX_OK) return rc;
  QvHead hd;
  if ((rc = qv_read_head(h_head,head_n,hd)) == DX_E_KEY)
    return dx_fail(ctx,DX_E_KEY,"not a .dexqv file (endian key 0x%04x)",(unsigned) hd.key);
  if (rc != DX_OK)
    return dx_fail(ctx,rc,"Could not read the coding header (Read_QVcoding) from the %zu head bytes",head_n);
  if (!hd.newv || hd.coding.flip)
    return dx_fail(ctx,DX_E_FORMAT,"%s image: byte ranges take images of the 0x55aa layout in the native byte "
                   "order; decode it whole with dx_undexqv_dev",hd.newv ? "a foreign-endian" : "an old-layout (key-less)");
  if (first != NULL) *first = (int64_t) hd.first;
  const int64_t A = std::max(a,(int64_t) hd.first), B = std::max(b,A);     // no entry starts inside the header
  const int64_t base = qv_range_base(A,buf_off), buf_end = buf_off + (int64_t) buf_n;
  if (a < 0 || a > b)
    return dx_fail(ctx,DX_E_ARG,"dx_undexqv_range_dev: bad range [%lld, %lld)",(long long) a,(long long) b);
  if (buf_off < 0 || base < buf_off || buf_end < b)
    return dx_fail(ctx,DX_E_ARG,"dx_undexqv_range_dev: the buffer holds the image bytes [%lld, %lld), the range [%lld, %lld) "
                   "needs at least [%lld, %lld)",(long long) buf_off,(long long) buf_end,(long long) a,(long long) b,
                   (long long) (A > 4096 ? A - 4096 : 0),(long long) B);
  cudaSetDevice(ctx->device);
  dx_arena_reset(ctx);
  if (ctx->qv_range == NULL) ctx->qv_range = new (std::nothrow) QvRange();
  if (ctx->qv_range == NULL) return DX_E_NOMEM;
  QvRange &R = *(QvRange *) ctx->qv_range;
  if ((rc = qv_range_setup(ctx,hd,upper,false,R)) != DX_OK) return rc;
  if (B == A)                                             // a range inside the header: no entry starts there
    rc = qv_range_decode(ctx,R,d_buf,0,buf_off,A,B);
  else
    rc = qv_range_decode(ctx,R,d_buf + (base - buf_off),(size_t) (buf_end - base),base,A,B);
  if (rc != DX_OK) return rc;
  ctx->qv_range_live = 1;
  return DX_OK;
}

extern "C" int dx_undexqv_range_chain(dx_ctx *ctx, int64_t cur_in, int32_t well_in, int64_t *cur_out, int32_t *well_out)
{ if (ctx == NULL || cur_out == NULL || well_out == NULL) return DX_E_ARG;
  if (!ctx->qv_range_live) return dx_fail(ctx,DX_E_ARG,"dx_undexqv_range_chain: no range decoded (dx_undexqv_range_dev)");
  QvRange &R = *(QvRange *) ctx->qv_range;
  if (cur_in < R.a)
    return dx_fail(ctx,DX_E_ARG,"dx_undexqv_range_chain: the chain position %lld lies in front of the range [%lld, %lld)",
                   (long long) cur_in,(long long) R.a,(long long) R.b);
  cudaSetDevice(ctx->device);
  const int rc = qv_range_chain(ctx,R,cur_in,well_in,cur_out,well_out);
  if (rc != DX_OK) ctx->qv_range_live = (rc == DX_E_CAP) ? 0 : ctx->qv_range_live;
  return rc;
}

extern "C" int dx_undexqv_range_text_dev(dx_ctx *ctx, uint8_t *d_out, size_t cap, size_t *out_len)
{ if (ctx == NULL || out_len == NULL) return DX_E_ARG;
  *out_len = 0;
  if (!ctx->qv_range_live) return dx_fail(ctx,DX_E_ARG,"dx_undexqv_range_text_dev: no range decoded (dx_undexqv_range_dev)");
  if (d_out == NULL && cap > 0) return dx_fail(ctx,DX_E_ARG,"dx_undexqv_range_text_dev: d_out is NULL");
  cudaSetDevice(ctx->device);
  int rc;
  if ((rc = qv_range_text(ctx,*(QvRange *) ctx->qv_range,d_out,cap,out_len)) != DX_OK) return rc;
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  return DX_OK;
}

// ------------------------------------------------------------------------------------------------
//  dx_undexqv_host as a pipeline: the image goes to the device in chunks (copy stream cs_in), every
//  chunk is a WINDOW -- a byte range, through the three steps above -- decoded as soon as it and its
//  successor have arrived (an entry may run over the boundary), and a window's text leaves for the
//  host (copy stream cs_out) while the next window is decoded: PCIe is busy in both directions and
//  the kernels hide behind the copies.  The chain carries its position, well number and text offset
//  from window to window.  Anything unusual (legacy layout, an entry longer than the bytes that have
//  arrived, a malformed image) -> *handled = false after the copies have drained, and the caller runs
//  the plain path on the complete image.
// ------------------------------------------------------------------------------------------------
static int pipe_setup(dx_ctx *ctx, int nev)
{ if (ctx->cs_in == NULL)  DX_CUDA(ctx,cudaStreamCreateWithFlags(&ctx->cs_in,cudaStreamNonBlocking));
  if (ctx->cs_out == NULL) DX_CUDA(ctx,cudaStreamCreateWithFlags(&ctx->cs_out,cudaStreamNonBlocking));
  while (ctx->npev < nev)
    { DX_CUDA(ctx,cudaEventCreateWithFlags(&ctx->pev[ctx->npev],cudaEventDisableTiming));
      ctx->npev++;
    }
  return DX_OK;
}

static int undexqv_pipe(dx_ctx *ctx, const uint8_t *h_in, size_t n, int upper, uint8_t *h_out, size_t cap,
                        size_t *out_len, bool *handled)
{ int rc;
  *handled = false;
  const size_t kMinChunk = ctx->route[DXR_PIPE_CHUNK] > 0 ? (size_t) ctx->route[DXR_PIPE_CHUNK] : (size_t) 32 << 20;
  if (n < 2*kMinChunk || kMinChunk < 16384 || ctx->route[DXR_SERIAL_IO] || ctx->route[DXR_DECODER] == 1 || ctx->route[DXR_NO_SPEC] ||
      ctx->route[DXR_NO_FAST] || ctx->keep_index) return DX_OK;
  QvHead hd;
  if (qv_read_head(h_in,2 + (n-2 < 300000 ? n-2 : 300000),hd) != DX_OK || hd.key != 0x55aa || hd.coding.flip) return DX_OK;
  // every window's decode launch lasts about as long as its longest entry (~2 ms with 60 000-position
  // entries), whatever else it holds: windows must stay large enough for the launch to hide behind the
  // text copy of the window before it
  int K = (int) (n / kMinChunk);
  if (K > 10) K = 10;                                     // measured on 2 GB: 4 windows 47 ms, 8-12 windows 42-44 ms, 16 45 ms, serial 54 ms
  const size_t chunk = round_up((n + (size_t) K - 1) / (size_t) K,(size_t) 4096);
  K = (int) ((n + chunk - 1) / chunk);
  cudaSetDevice(ctx->device);
  if ((rc = pipe_setup(ctx,2*K + 2)) != DX_OK) return rc;
  if ((rc = ensure_io(ctx,&ctx->io_in,&ctx->io_in_cap,n)) != DX_OK) return rc;
  if ((rc = ensure_io(ctx,&ctx->io_out,&ctx->io_out_cap,cap)) != DX_OK) return rc;
  dx_arena_reset(ctx);
  const uint8_t *d_in = ctx->io_in;
  uint8_t *d_out = ctx->io_out;
  // all chunks on their way; event k = chunk k has arrived
  for (int k = 0; k < K; k++)
    { const size_t a = (size_t) k*chunk, b = (a + chunk < n) ? a + chunk : n;
      DX_CUDA(ctx,cudaMemcpyAsync(ctx->io_in + a,h_in + a,b - a,cudaMemcpyHostToDevice,ctx->cs_in));
      DX_CUDA(ctx,cudaEventRecord(ctx->pev[k],ctx->cs_in));
    }

  auto drain = [&]() { cudaStreamSynchronize(ctx->cs_in); cudaStreamSynchronize(ctx->cs_out);
                       cudaStreamSynchronize(ctx->stream); };

  QvRange R;
  if ((rc = qv_range_setup(ctx,hd,upper,true,R)) != DX_OK) { drain(); return rc; }

  int64_t cur = (int64_t) hd.first;        // image offset of the next entry (chain position)
  int32_t well = 0;
  size_t  tbase = 0;                       // text bytes of the windows before this one
  for (int k = 0; k < K; k++)
    { const size_t wa = (size_t) k*chunk, wb = (wa + chunk < n) ? wa + chunk : n;      // entries starting in [wa, wb)
      const size_t avail = ((size_t) (k + 2)*chunk < n) ? (size_t) (k + 2)*chunk : n;  // bytes on the device
      DX_CUDA(ctx,cudaStreamWaitEvent(ctx->stream,ctx->pev[(k + 1 < K) ? k + 1 : k],0));
      const int64_t a = std::max((int64_t) wa,(int64_t) hd.first), b = std::max((int64_t) wb,a);
      const int64_t base = qv_range_base(a,0);
      if ((rc = qv_range_decode(ctx,R,d_in + base,avail - (size_t) base,base,a,b)) != DX_OK) { drain(); return rc; }
      int64_t stop = 0;
      int32_t wlast = 0;
      rc = qv_range_chain(ctx,R,cur,well,&stop,&wlast);
      if (rc == DX_E_CAP || rc == DX_E_TRUNC || rc == DX_E_FORMAT) { drain(); return DX_OK; }    // the plain path decides
      if (rc != DX_OK) { drain(); return rc; }
      cur = stop; well = wlast;
      if (R.ent.empty()) continue;
      size_t wtext = 0;
      if ((rc = qv_range_text(ctx,R,d_out + tbase,cap - tbase,&wtext)) != DX_OK)
        { drain(); return (rc == DX_E_CAP) ? dx_fail(ctx,DX_E_CAP,"output needs more than %zu bytes",cap) : rc; }
      // this window's text leaves while the next window is decoded
      DX_CUDA(ctx,cudaEventRecord(ctx->pev[K + k],ctx->stream));
      DX_CUDA(ctx,cudaStreamWaitEvent(ctx->cs_out,ctx->pev[K + k],0));
      DX_CUDA(ctx,cudaMemcpyAsync(h_out + tbase,d_out + tbase,wtext,cudaMemcpyDeviceToHost,ctx->cs_out));
      tbase += wtext;
    }
  drain();
  if (cur != (int64_t) n) return DX_OK;                              // (the plain path reports what is wrong)
  *out_len = tbase;
  *handled = true;
  return DX_OK;
}

extern "C" int dx_undexqv_host(dx_ctx *ctx, const uint8_t *h_in, size_t n, int upper,
                               uint8_t *h_out, size_t cap, size_t *out_len)
{ if (ctx == NULL || h_in == NULL || h_out == NULL || out_len == NULL) return DX_E_ARG;
  int rc;
  { bool handled = false;
    if ((rc = undexqv_pipe(ctx,h_in,n,upper,h_out,cap,out_len,&handled)) != DX_OK) return rc;
    if (handled) return DX_OK;
  }
  if ((rc = stage_in(ctx,h_in,n)) != DX_OK) return rc;
  if ((rc = ensure_io(ctx,&ctx->io_out,&ctx->io_out_cap,cap)) != DX_OK) return rc;
  if ((rc = dx_undexqv_dev(ctx,ctx->io_in,n,upper,ctx->io_out,cap,out_len,NULL,0,0)) != DX_OK) return rc;
  return stage_out(ctx,h_out,*out_len);
}
