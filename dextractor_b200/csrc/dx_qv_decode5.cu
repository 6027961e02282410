// dx_qv_decode5.cu -- parallel .dexqv entry decoder, one WARP per entry (the one the library uses).
//
// Replaces Decode / Decode_Run (reference QV.c:510-691) + Packed_Length / Unpack_Tag
// (QV.c:823-847) + the per-entry text output of undexqv.c:182-207.
//
// A persistent grid of one 32-warp CTA per SM; every warp pulls entries from a ticket counter and
// decodes the entry's streams one after the other, 32 subsequences of 256 bits at a time.  All
// synchronisation is inside the warp (shuffles), so no warp ever waits at a CTA barrier and
// ~4700 entries are in flight on the chip.  The stream's 12-bit decode tables for all four
// Huffman streams stay resident in shared memory (64 KB per CTA, loaded once).
//
//   0. the window's words are staged in shared memory as overlapping 64-bit pairs (word j in the
//      high half, word j+1 in the low half), already shifted to the stream's byte alignment: the
//      32 bits at ANY bit position are one 64-bit shared load and one funnel shift.  Each lane
//      owns a region of 9 pairs (stride 9: conflict-free banks).  Only as many lanes as the code
//      lengths predict for the symbols still to come are active; whatever is left of the stream
//      simply becomes the next window;
//   1. lane i decodes from bit 256*i (a guess) to the first code boundary at or past bit
//      256*(i+1), its EXIT, counting symbols (plain streams: up to two symbols per lookup);
//   2. rounds: a lane whose start differs from its predecessor's exit walks two fingers, one from
//      its old start and one from the new one, always advancing the one behind by a single
//      symbol, until they meet: from there on both paths are the same, so exit and counts follow
//      by arithmetic.  Lane 0 starts at the true position, so at the fix point every start is a
//      true code boundary (induction over the lanes);
//   3. a warp scan of the symbol counts places every subsequence in the output line and finds the
//      subsequence in which the rlen-th symbol -- hence the stream -- ends; the stream's length in
//      the file follows from the position of its last item ((p_last+47)>>5 words, the
//      reference's refill rule, QV.c:537-551);
//   4. every lane decodes its subsequence once more, now producing text: run-length streams
//      scatter their non-run symbols into a line pre-filled with the run character, plain streams
//      go through a per-warp shared-memory stage that is flushed with aligned 32-bit stores.
// Speculation only costs time: nothing is written before the fix point is reached.

#include <stdio.h>
#include <stdlib.h>
#include "dx_internal.h"
#include "dx_common.cuh"

namespace {

constexpr int kWarps    = 32;
constexpr int kThreads  = kWarps * 32;
constexpr int kS        = 256;                  // bits per subsequence
constexpr int kSW       = kS / 32;              // words per subsequence
constexpr int kRegion   = kSW + 1;              // 64-bit pairs per lane (one look-ahead pair)
constexpr int kStage    = 2560;                 // bytes of a warp's output stage
constexpr int kTail     = 24;                   // longest single step (16-bit code + 8-bit literal)
constexpr int kFingerBudget = 24;               // two-finger steps per lane beyond which the stream's code counts as slow to synchronise

struct Dec5Args
{ const uint8_t *in;
  int64_t        n;
  const QvDecTables4 *tab;
  int32_t        delchar, subchar, upper, write;   // write: 0 walk, 1 text + header, 2 lines only
                                                   //        (speculative, per-entry status), 3 text +
                                                   //        header in place AND per-entry status
  int64_t        count;
  const int64_t *start;        // first stream byte of each entry (after beg/end/qv)
  const int32_t *rlen;
  const QvDecEntry *ent;       // write mode: output placement
  const int64_t *toff;         // write == 2 without ent: where the entry's lines go
  const char    *prefix; int32_t plen;
  uint8_t       *out;
  int64_t       *soff;         // [count][6] or NULL
  int32_t       *status;       // [count] (walk) or [1] (decode)
  const int64_t *limit;        // per entry: first byte the entry may not reach (NULL: the image end)
  const int32_t *order;        // ticket -> entry (long entries first), NULL: identity
  const int64_t *endat;        // per entry: the byte its streams must end at (known offsets), NULL: any
  unsigned long long *ticket;
  unsigned long long *dbg;     // optional counters [table][0 rounds, 1 windows, 2 streams, 3 restarts]
};

struct WarpMem
{ uint64_t bits[32*kRegion];                // pair 9*lane + k = stream words 8*lane+k, 8*lane+k+1
  uint32_t stage[kStage/4 + 4];
};

struct Shared5
{ uint32_t tab[4][4096];                    // del, ins, mrg, sub: one multi table or run|sym u16 tables
  WarpMem  w[kWarps];
};

extern __shared__ __align__(16) uint8_t dx_dec5_smem[];

// the 32 stream bits that start at window-relative bit `pos` (D already offset by the lane)
__device__ __forceinline__ uint32_t win32(const uint64_t *D, uint32_t pos)
{ const uint64_t v = D[pos >> 5];
  return __funnelshift_l((uint32_t) v,(uint32_t) (v >> 32),pos);
}

// codes longer than 12 bits: sym | len << 8, len 0 = no code maps here
__device__ __forceinline__ uint32_t lookup_long(const QvDecTables2 *t, int k, uint32_t w16)
{ uint32_t e = __ldg(&t->prim[k][w16 >> 5]);
  if (e & 0x8000u)
    e = __ldg(&t->sub[k][(e & 0x7fffu)*32u + (w16 & 31u)]);
  return e;
}

// ... as an entry of the plain-stream table (see QvDecTables4)
__device__ __noinline__ uint32_t long_entry(const QvDecTables2 *t, int k, uint32_t w, uint32_t *bad)
{ const uint32_t f = lookup_long(t,k,w >> 16);
  uint32_t len = (f >> 8) & 31u;
  const uint32_t c = f & 0xffu;
  if (len == 0) { len = 1; *bad = 1; }
  if (t->type[k] == 2 && c == 255u)
    return (len + 8u) | (1u << 5) | 0x80u | (len << 8) | (255u << 16);
  return len | (1u << 5) | (len << 8) | (c << 16);
}

// ... as an entry of a single-symbol table: sym | len << 8, len >= 1
__device__ __noinline__ uint32_t long_single(const QvDecTables2 *t, int k, uint32_t w, uint32_t *bad)
{ uint32_t f = lookup_long(t,k,w >> 16) & 0x1fffu;
  if ((f >> 8) == 0u) { f |= 0x100u; *bad = 1; }
  return f;
}

// the warp fills dst[0..n) with byte c (any alignment)
__device__ __forceinline__ void fill_line(uint8_t *dst, uint32_t c, uint32_t n, uint32_t lane)
{ uint32_t head = (16u - (uint32_t) (reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u;
  if (head > n) head = n;
  if (lane < head) dst[lane] = (uint8_t) c;
  const uint32_t nvec = (n - head) >> 4;
  const uint32_t q = c * 0x01010101u;
  const uint4 v = make_uint4(q,q,q,q);
  uint8_t *body = dst + head;
  for (uint32_t i = lane; i < nvec; i += 32) dx_stg16(body + (size_t) i*16,v);
  const uint32_t done = head + nvec*16u;
  if (lane < n - done) dst[done + lane] = (uint8_t) c;
}

// lane < nact stages its region: stream words 8*lane .. 8*lane+9 of the window that starts at p
__device__ __forceinline__ void stage_window(const Dec5Args &a, uint64_t *bits, const uint8_t *p,
                                             uint32_t lane, uint32_t nact)
{ if (lane < nact)
    { const uintptr_t A = reinterpret_cast<uintptr_t>(p) + 32u*lane;
      const uint32_t *al = reinterpret_cast<const uint32_t *>(A & ~(uintptr_t) 3);
      const uint32_t sh = (uint32_t) (A & 3) * 8;
      const uint32_t *endw = reinterpret_cast<const uint32_t *>(
                               (reinterpret_cast<uintptr_t>(a.in + a.n) + 3) & ~(uintptr_t) 3);
      uint32_t x[kRegion + 2];
#pragma unroll
      for (int k = 0; k < kRegion + 2; k++) x[k] = (al + k < endw) ? __ldg(al + k) : 0u;
#pragma unroll
      for (int k = 0; k < kRegion; k++)
        { const uint32_t w0 = __funnelshift_r(x[k],x[k+1],sh), w1 = __funnelshift_r(x[k+1],x[k+2],sh);
          bits[kRegion*lane + k] = ((uint64_t) w0 << 32) | w1;
        }
    }
  __syncwarp();
}

// multi entry: bits 0-4 total length (escape: code + 8 literal bits), 5-6 symbols (1|2),
// bit 7 escape, 8-12 length of the first code, 16-23 first symbol, 24-31 second symbol; 0 = long
#define DX_E_LEN(e)   ((e) & 31u)
#define DX_E_N(e)     (((e) >> 5) & 3u)
#define DX_E_LEN0(e)  (((e) >> 8) & 31u)
#define DX_E_LEN1(e)  (((e) & 0x40u) ? DX_E_LEN0(e) : DX_E_LEN(e))      /* one symbol only */

struct StreamOut { uint32_t bytes, kept, bad; };

// Decode one stream of `rlen` symbols that starts at byte `so`, by one warp.  bytes = what the
// stream occupies in the file; kept = symbol items != rc.  `dst` != NULL: the line is written.
template <bool RUN>
__device__ __noinline__ StreamOut decode_stream(const Dec5Args &a, int slot, int64_t so, int32_t rlen,
                                                int symtab, int runtab, int32_t rci, uint8_t *dst,
                                                int64_t budget)
{ Shared5 &sm = *reinterpret_cast<Shared5 *>(dx_dec5_smem);
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  StreamOut res; res.bytes = 0; res.kept = 0; res.bad = 0;
  if (rlen <= 0)
    { if (dst != NULL && lane == 0) dst[0] = '\n';
      return res;
    }
  const QvDecTables2 *t2 = &a.tab->t2;
  const bool esc = (t2->type[symtab] == 2);
  const uint32_t rc = (uint32_t) rci;                 // 0xffffffff for plain streams
  const uint32_t base = lane * kS, lim = base + kS;
  const float abits = a.tab->abits[symtab] * 1.2f;
  WarpMem &wm = sm.w[warp];
  const uint64_t *D = wm.bits + lane;                 // pair index = (pos >> 5) + lane
  const uint32_t *mt = sm.tab[slot];
  const uint16_t *rt = reinterpret_cast<const uint16_t *>(sm.tab[slot]), *st = rt + 4096;
  uint32_t done = 0;                                  // symbols placed by earlier windows
  uint32_t carry = 0;                                 // start state of lane 0 (window relative)
  uint32_t wword = 0;                                 // first stream word of the window
  uint32_t bd = 0, sp = 0, ksum = 0;     // bd: malformed stream seen by the final pass; sp: speculation only
  bool redecode = false;                 // plain streams: re-synchronise by decoding again (set by the first slow window)
  if (RUN && dst != NULL) fill_line(dst,rc,(uint32_t) rlen,lane);

  while (true)
    { const uint32_t remaining = (uint32_t) rlen - done;
      uint32_t nact = (uint32_t) ((float) remaining * abits * (1.0f/kS)) + 2u;
      if (nact > 32u) nact = 32u;
      const bool active = (lane < nact);
      __syncwarp();
      stage_window(a,wm.bits,a.in + so + (int64_t) wword*4,lane,nact);

      // ---- round 0: from the guessed start to the exit --------------------------------------------
      // state = bit position << 1 | parity (1: a run item was read, its symbol item comes next)
      uint32_t mystart = (lane == 0) ? carry : (base << 1);
      uint32_t myexit = 0, n = 0, nk = 0;
      if (active)
        { uint32_t pos = mystart >> 1, cnt = 0, kept = 0;
          if (RUN)
            { uint32_t par = mystart & 1u;
              while (pos < lim)
                { if (par == 0)
                    { uint32_t w = win32(D,pos);
                      uint32_t e = rt[w >> 20];
                      if (e == 0u) e = long_single(t2,runtab,w,&sp);
                      uint32_t r = e & 0xffu;
                      pos += e >> 8;
                      if (r == 255u) { r = win32(D,pos) >> 16; pos += 16; }
                      cnt += r;
                      par = 1;
                      if (pos >= lim) break;
                    }
                  uint32_t w = win32(D,pos);
                  uint32_t e = st[w >> 20];
                  if (e == 0u) e = long_single(t2,symtab,w,&sp);
                  uint32_t c = e & 0xffu;
                  pos += e >> 8;
                  if (esc && c == 255u) { c = win32(D,pos) >> 24; pos += 8; }
                  cnt += 1;
                  kept += (c != rc);
                  par = 0;
                }
              myexit = (pos << 1) | par;
            }
          else
            { const uint32_t limf = lim - kTail;      // below it no step can reach the limit
              while (pos < limf)
                { const uint32_t w = win32(D,pos);
                  uint32_t e = mt[w >> 20];
                  if (e == 0u) e = long_entry(t2,symtab,w,&sp);
                  pos += DX_E_LEN(e);
                  cnt += DX_E_N(e);
                }
              while (pos < lim)                       // one symbol at a time: the exit is the FIRST
                { const uint32_t w = win32(D,pos);    // code boundary at or past the limit
                  uint32_t e = mt[w >> 20];
                  if (e == 0u) e = long_entry(t2,symtab,w,&sp);
                  pos += DX_E_LEN1(e);
                  cnt += 1;
                }
              myexit = pos << 1;
            }
          n = cnt; nk = kept;
        }

      // ---- rounds: adopt the predecessor's exit; two fingers until the old path is met ----------
      uint32_t rounds = 0, restarts = 0, slow = 0;
      bool giveup = false;
      while (true)
        { int changed = 0;
          uint32_t want = __shfl_up_sync(DX_FULL,myexit,1);
          if (!active || lane == 0) want = mystart;
          if (want != mystart)
            { uint32_t pa = mystart >> 1, pb = want >> 1, ca = 0, cb = 0, ka = 0, kb = 0;
              restarts++;
              if (RUN)
                { uint32_t qa = mystart & 1u, qb = want & 1u;
                  while (!(pa == pb && qa == qb) && min(pa,pb) < lim)
                    { const bool fa = (pa <= pb);
                      uint32_t pos = fa ? pa : pb, par = fa ? qa : qb, dc, dk = 0;
                      if (par == 0)
                        { uint32_t w = win32(D,pos);
                          uint32_t e = rt[w >> 20];
                          if (e == 0u) e = long_single(t2,runtab,w,&sp);
                          dc = e & 0xffu;
                          pos += e >> 8;
                          if (dc == 255u) { dc = win32(D,pos) >> 16; pos += 16; }
                          par = 1;
                        }
                      else
                        { uint32_t w = win32(D,pos);
                          uint32_t e = st[w >> 20];
                          if (e == 0u) e = long_single(t2,symtab,w,&sp);
                          uint32_t c = e & 0xffu;
                          pos += e >> 8;
                          if (esc && c == 255u) { c = win32(D,pos) >> 24; pos += 8; }
                          dc = 1; dk = (c != rc);
                          par = 0;
                        }
                      if (fa) { pa = pos; qa = par; ca += dc; ka += dk; }
                      else    { pb = pos; qb = par; cb += dc; kb += dk; }
                    }
                  if (pa == pb && qa == qb) { n += cb - ca; nk += kb - ka; }
                  else { n = cb; nk = kb; myexit = (pb << 1) | qb; changed = 1; }
                }
              else if (redecode)
                { // a code that synchronises slowly: two fingers would keep the whole warp waiting for
                  // its unluckiest lane, so decode the subsequence again at full speed instead
                  uint32_t pos = want >> 1, cnt = 0;
                  const uint32_t limf = lim - kTail;
                  while (pos < limf)
                    { const uint32_t w = win32(D,pos);
                      uint32_t e = mt[w >> 20];
                      if (e == 0u) e = long_entry(t2,symtab,w,&sp);
                      pos += DX_E_LEN(e);
                      cnt += DX_E_N(e);
                    }
                  while (pos < lim)
                    { const uint32_t w = win32(D,pos);
                      uint32_t e = mt[w >> 20];
                      if (e == 0u) e = long_entry(t2,symtab,w,&sp);
                      pos += DX_E_LEN1(e);
                      cnt += 1;
                    }
                  n = cnt;
                  if ((pos << 1) != myexit) { myexit = pos << 1; changed = 1; }
                }
              else
                { uint32_t steps = 0;
                  while (pa != pb && min(pa,pb) < lim)
                    { const bool fa = (pa < pb);
                      const uint32_t pos = fa ? pa : pb;
                      const uint32_t w = win32(D,pos);
                      uint32_t e = mt[w >> 20];
                      if (e == 0u) e = long_entry(t2,symtab,w,&sp);
                      const uint32_t np = pos + DX_E_LEN1(e);
                      if (fa) { pa = np; ca++; } else { pb = np; cb++; }
                      steps++;
                    }
                  if (steps > kFingerBudget) slow = 1;
                  if (pa == pb) n += cb - ca;
                  else { n = cb; myexit = pb << 1; changed = 1; }
                }
              mystart = want;
            }
          rounds++;
          if (!__any_sync(DX_FULL,changed)) break;
          if (a.limit != NULL && rounds >= 12u) { giveup = true; break; }
        }
      if (!RUN && !redecode && __any_sync(DX_FULL,slow != 0)) redecode = true;
      if (giveup)                     // speculative modes: this does not look like a code stream (a false
        { bd = 1;                     // candidate); a true entry given up here is found by the slow path
          res.bytes = wword*4u;
          break;
        }
      if (a.dbg != NULL)
        { if (lane == 0) { atomicAdd(&a.dbg[symtab*4],(unsigned long long) rounds);
                           atomicAdd(&a.dbg[symtab*4+1],1ull); }
          if (restarts) atomicAdd(&a.dbg[symtab*4+3],(unsigned long long) restarts);
        }

      // ---- place the subsequences ---------------------------------------------------------------
      const uint32_t inc = dx_warp_incl_sum(n,lane);
      const uint32_t total = __shfl_sync(DX_FULL,inc,31);
      const uint32_t before = inc - n;
      const bool ends_here = (total >= remaining);
      const bool owner = ends_here && before < remaining && remaining <= before + n;
      uint32_t need = 0;
      if (before < remaining) need = min(n,remaining - before);

      // ---- final decode: text, and for the owner of the rlen-th symbol the end of the stream ----
      const bool wr = (dst != NULL);
      const uint32_t outn = min(total,remaining);
      const bool staged = wr && !RUN && outn <= (uint32_t) kStage;
      uint32_t last = 0, kfin = 0;
      if (need > 0 && (wr || owner))
        { uint8_t *p;
          if (staged) p = reinterpret_cast<uint8_t *>(wm.stage) + before;
          else        p = dst + done + before;
          uint32_t pos = mystart >> 1, cnt = 0;
          if (RUN)
            { uint32_t par = mystart & 1u;
              while (cnt < need)
                { if (par == 0)
                    { uint32_t w = win32(D,pos);
                      uint32_t e = rt[w >> 20];
                      if (e == 0u) e = long_single(t2,runtab,w,&bd);
                      uint32_t r = e & 0xffu;
                      last = pos;
                      pos += e >> 8;
                      if (r == 255u) { r = win32(D,pos) >> 16; last = pos; pos += 16; }
                      if (r > need - cnt) { r = need - cnt; bd = 1; }
                      cnt += r; p += r;
                      par = 1;
                      if (cnt >= need) break;
                    }
                  uint32_t w = win32(D,pos);
                  uint32_t e = st[w >> 20];
                  if (e == 0u) e = long_single(t2,symtab,w,&bd);
                  uint32_t c = e & 0xffu;
                  last = pos;
                  pos += e >> 8;
                  if (esc && c == 255u) { c = win32(D,pos) >> 24; last = pos; pos += 8; }
                  if (wr) *p = (uint8_t) c;
                  p++; cnt++;
                  kfin += (c != rc);
                  par = 0;
                }
            }
          else
            { // all lookups but the last ones: up to two symbols each, nothing to check
              while (cnt + 2u < need)
                { const uint32_t w = win32(D,pos);
                  uint32_t e = mt[w >> 20];
                  if (e == 0u) e = long_entry(t2,symtab,w,&bd);
                  uint32_t c0 = (e >> 16) & 0xffu;
                  if (e & 0x80u) c0 = (w << DX_E_LEN0(e)) >> 24;      // the literal after the escape
                  if (wr)
                    { p[0] = (uint8_t) c0;
                      if (e & 0x40u) p[1] = (uint8_t) (e >> 24);
                    }
                  pos += DX_E_LEN(e);
                  p   += DX_E_N(e);
                  cnt += DX_E_N(e);
                }
              // the last one or two symbols, one at a time: `last` is the position of the last item
              // (the literal of an escape)
              while (cnt < need)
                { const uint32_t w = win32(D,pos);
                  uint32_t e = mt[w >> 20];
                  if (e == 0u) e = long_entry(t2,symtab,w,&bd);
                  uint32_t c0 = (e >> 16) & 0xffu;
                  const uint32_t l0 = DX_E_LEN0(e);
                  last = pos;
                  if (e & 0x80u) { c0 = (w << l0) >> 24; last = pos + l0; }
                  if (wr) p[0] = (uint8_t) c0;
                  pos += (e & 0x80u) ? l0 + 8u : l0;
                  p++; cnt++;
                }
            }
        }
      if (RUN && symtab == 0)
        { uint32_t contrib = 0;
          if (owner) contrib = kfin;
          else if (need == n && n > 0) contrib = nk;
          ksum += dx_warp_sum(contrib);
        }
      if (staged)
        { __syncwarp();
          dx_warp_copy_out(dst + done,wm.stage,outn,lane);
        }
      if (ends_here)
        { const uint32_t who = __ffs(__ballot_sync(DX_FULL,owner)) - 1;
          const uint32_t endw = (wword*32u + last + 47u) >> 5;     // reference refill rule (QV.c:537-551)
          res.bytes = __shfl_sync(DX_FULL,endw,who & 31u) * 4u;
          break;
        }
      done  += total;
      carry  = __shfl_sync(DX_FULL,myexit,nact-1) - ((nact*kS) << 1);
      wword += nact*kSW;
      if (so + (int64_t) wword*4 > budget + 8)           // ran off the image / its budget: corrupt or false start
        { bd = 1;
          res.bytes = wword*4u;
          break;
        }
    }
  __syncwarp();
  if (a.dbg != NULL && lane == 0) atomicAdd(&a.dbg[symtab*4+2],1ull);
  if (dst != NULL && lane == 0) dst[rlen] = '\n';
  res.kept = ksum;
  res.bad  = __any_sync(DX_FULL,bd != 0);
  return res;
}

// tag line by one warp: positions whose deletion QV is the run character get 'n', the others the
// next packed tag (Unpack_Tag, QV.c:837-847); the del line is read back from global memory
__device__ __noinline__ void write_tags(const Dec5Args &a, const uint8_t *del, const uint8_t *packed,
                                        int32_t rlen, uint8_t *dst)
{ Shared5 &sm = *reinterpret_cast<Shared5 *>(dx_dec5_smem);
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  uint32_t *stw = sm.w[warp].stage;
  uint8_t  *stb = reinterpret_cast<uint8_t *>(stw);
  const uint32_t caseoff = a.upper ? 32u : 0u;
  const uint32_t nn = ('n' - caseoff) * 0x01010101u;
  uint32_t rank = 0;
  for (int32_t p0 = 0; p0 < rlen; p0 += 512)
    { const int32_t p = p0 + (int32_t) lane*16;
      const int cnt = max(0,min(16,rlen - p));
      uint32_t m = 0;
      if (cnt > 0)
        { if (a.delchar < 0) m = (1u << cnt) - 1u;
          else
            { // the lane's 16 bytes of the del line (any alignment) from five aligned words; only words
              // that hold a byte of the line are read (the last of them ends at most three bytes
              // behind it: the newline and the tag line are there)
              const uintptr_t A = reinterpret_cast<uintptr_t>(del + p);
              const uint32_t *al = reinterpret_cast<const uint32_t *>(A & ~(uintptr_t) 3);
              const uint32_t *endw = reinterpret_cast<const uint32_t *>(
                                       (reinterpret_cast<uintptr_t>(del + rlen) + 3) & ~(uintptr_t) 3);
              const uint32_t sh = (uint32_t) (A & 3) * 8;
              uint32_t x[5];
#pragma unroll
              for (int k = 0; k < 5; k++) x[k] = (al + k < endw) ? __ldcg(al + k) : 0u;
              const uint4 d = make_uint4(__funnelshift_r(x[0],x[1],sh),__funnelshift_r(x[1],x[2],sh),
                                         __funnelshift_r(x[2],x[3],sh),__funnelshift_r(x[3],x[4],sh));
              m = ~dx_eq_mask16(d,(uint32_t) a.delchar) & ((1u << cnt) - 1u);
            }
        }
      const uint32_t c = __popc(m);
      const uint32_t inc = dx_warp_incl_sum(c,lane);
      uint32_t r = rank + inc - c;
      rank += __shfl_sync(DX_FULL,inc,31);
      stw[4*lane] = nn; stw[4*lane+1] = nn; stw[4*lane+2] = nn; stw[4*lane+3] = nn;
      while (m)
        { const int k = __ffs(m) - 1; m &= m - 1;
          const uint32_t byte = __ldg(packed + (r >> 2));
          const uint32_t ch = (0x74676361u >> (8*((byte >> (6 - 2*(r & 3))) & 3u))) & 0xffu;
          stb[16*lane + k] = (uint8_t) (ch - caseoff);
          r++;
        }
      __syncwarp();
      dx_warp_copy_out(dst + p0,stw,(uint32_t) min(512,rlen - p0),lane);
      __syncwarp();
    }
  if (lane == 0) dst[rlen] = '\n';
}

__device__ int fmt_int5(uint8_t *p, int32_t v)
{ char tmp[12];
  int  k = 0, len = 0;
  uint32_t u = (v < 0) ? (uint32_t) (-(int64_t) v) : (uint32_t) v;
  if (v < 0) p[len++] = '-';
  do { tmp[k++] = (char) ('0' + u % 10); u /= 10; } while (u);
  while (k) p[len++] = (uint8_t) tmp[--k];
  return len;
}

__global__ void __launch_bounds__(kThreads,1)
k_qv_decode5(Dec5Args a)
{ Shared5 &sm = *reinterpret_cast<Shared5 *>(dx_dec5_smem);
  const uint32_t lane = threadIdx.x & 31u;

  // resident tables: slot 0 del, 1 ins, 2 mrg, 3 sub
  { const QvDecTables4 *T = a.tab;
    for (int s = 0; s < 4; s++)
      { const int symtab = (s == 0) ? 0 : (s == 1) ? 2 : (s == 2) ? 3 : 4;
        const int runtab = (s == 0) ? 1 : 5;
        const bool run = (s == 0 && a.delchar >= 0) || (s == 3 && a.subchar >= 0);
        if (run)
          { const uint32_t *gr = reinterpret_cast<const uint32_t *>(T->single[runtab]);
            const uint32_t *gs = reinterpret_cast<const uint32_t *>(T->single[symtab]);
            for (int j = threadIdx.x; j < 2048; j += kThreads)
              { sm.tab[s][j] = __ldg(gr + j); sm.tab[s][2048 + j] = __ldg(gs + j); }
          }
        else
          for (int j = threadIdx.x; j < 4096; j += kThreads) sm.tab[s][j] = __ldg(T->multi[symtab] + j);
      }
  }
  __syncthreads();

  while (true)
    { unsigned long long tk = 0;
      if (lane == 0) tk = atomicAdd(a.ticket,1ull);
      const int64_t t = (int64_t) __shfl_sync(DX_FULL,tk,0);
      if (t >= a.count) break;
      const int64_t e = (a.order != NULL) ? (int64_t) a.order[t] : t;
      const int64_t lim = (a.limit != NULL) ? a.limit[e] : a.n;
      const int32_t L = a.rlen[e];
      int64_t at = a.start[e];
      int64_t o[6];
      uint8_t *line = NULL;
      if (L < 0)                                             // ruled out by the planner: nothing is written
        { if (lane == 0 && a.write != 1) a.status[e] = 1;
          continue;
        }
      if (a.write == 2 && a.ent == NULL)
        line = a.out + a.toff[e];
      else if (a.write)
        { const QvDecEntry en = a.ent[e];
          line = a.out + en.text_off;
          if (lane == 0 && (a.write & 1))
            { uint8_t *h = a.out + en.out_off;          // "%s/%d/%d_%d RQ=0.%d\n" (undexqv.c:182)
              int hl = 0;
              for (int k = 0; k < a.plen; k++) h[hl++] = (uint8_t) a.prefix[k];
              h[hl++] = '/'; hl += fmt_int5(h+hl,en.well);
              h[hl++] = '/'; hl += fmt_int5(h+hl,en.beg);
              h[hl++] = '_'; hl += fmt_int5(h+hl,en.end);
              const char *rq = " RQ=0.";
              for (int k = 0; k < 6; k++) h[hl++] = (uint8_t) rq[k];
              hl += fmt_int5(h+hl,en.qv);
              h[hl++] = '\n';
            }
        }
      const int64_t stride = (int64_t) L + 1;
      uint32_t bad = 0;
      StreamOut r;
      for (int k = 0; k < 6; k++) o[k] = at;

      // a candidate that turns out not to be an entry (speculative modes) is dropped at the first sign
      do
        { o[0] = at;
          if (a.delchar >= 0) r = decode_stream<true >(a,0,at,L,0,1,a.delchar,line,lim);
          else                r = decode_stream<false>(a,0,at,L,0,1,-1,line,lim);
          at += r.bytes; bad |= r.bad;
          o[1] = at;
          if (bad && a.write != 1) break;
          const uint32_t clen = (a.delchar < 0) ? (uint32_t) L : r.kept;
          if (a.write && at + (int64_t) ((clen + 3) >> 2) <= a.n)
            { __syncwarp();                                      // the del line is complete in global memory
              write_tags(a,line,a.in + at,L,line + stride);
            }
          at += (clen + 3) >> 2;
          o[2] = at;
          r = decode_stream<false>(a,1,at,L,2,0,-1,a.write ? line + 2*stride : NULL,lim);
          at += r.bytes; bad |= r.bad;
          o[3] = at;
          if (bad && a.write != 1) break;
          r = decode_stream<false>(a,2,at,L,3,0,-1,a.write ? line + 3*stride : NULL,lim);
          at += r.bytes; bad |= r.bad;
          o[4] = at;
          if (bad && a.write != 1) break;
          if (a.subchar >= 0) r = decode_stream<true >(a,3,at,L,4,5,a.subchar,a.write ? line + 4*stride : NULL,lim);
          else                r = decode_stream<false>(a,3,at,L,4,5,-1,a.write ? line + 4*stride : NULL,lim);
          at += r.bytes; bad |= r.bad;
          o[5] = at;
        }
      while (false);
      if (lane == 0)
        { if (at > lim) bad = 1;
          if (a.endat != NULL && at != a.endat[e]) bad = 1;     // the streams do not fill the entry
          if (a.soff != NULL)
            for (int k = 0; k < 6; k++) a.soff[e*6 + k] = o[k];
          if (a.write == 1) { if (bad) atomicExch(a.status,1); }
          else a.status[e] = (int32_t) bad;
        }
      __syncwarp();
    }
}


// ---- assembling the output of a speculative decode -------------------------------------------------
// The entries of a .dexqv whose boundaries had to be discovered are decoded BEFORE the chain of
// entries is verified, into a scratch image whose layout depends on the candidates alone (lines
// only).  Once the host has accepted the chain, one warp per entry writes the header line
// (undexqv.c:182) and moves the five lines to their place in the text.
struct AsmArgs
{ const uint8_t *tmp; const uint8_t *tmp_end16;
  const QvDecEntry *ent; const int64_t *src; int64_t count;
  const char *prefix; int32_t plen;
  uint8_t *out;
};

__global__ void __launch_bounds__(256)
k_qv_assemble(AsmArgs a)
{ const uint32_t lane = threadIdx.x & 31u;
  const int64_t nwarp = ((int64_t) gridDim.x * blockDim.x) >> 5;
  for (int64_t e = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5; e < a.count; e += nwarp)
    { const int64_t so = a.src[e];
      if (so < 0) continue;                                  // decoded in place by k_qv_decode5
      const QvDecEntry en = a.ent[e];
      if (lane == 0)
        { uint8_t *h = a.out + en.out_off;
          int hl = 0;
          for (int k = 0; k < a.plen; k++) h[hl++] = (uint8_t) a.prefix[k];
          h[hl++] = '/'; hl += fmt_int5(h+hl,en.well);
          h[hl++] = '/'; hl += fmt_int5(h+hl,en.beg);
          h[hl++] = '_'; hl += fmt_int5(h+hl,en.end);
          const char *rq = " RQ=0.";
          for (int k = 0; k < 6; k++) h[hl++] = (uint8_t) rq[k];
          hl += fmt_int5(h+hl,en.qv);
          h[hl++] = '\n';
        }
      const int64_t n = 5*((int64_t) en.end - en.beg + 1);
      uint8_t *dst = a.out + en.text_off;
      const uint8_t *src = a.tmp + so;
      int64_t head = (16 - (int64_t) (reinterpret_cast<uintptr_t>(dst) & 15)) & 15;
      if (head > n) head = n;
      if ((int64_t) lane < head) dst[lane] = src[lane];
      const int64_t nvec = (n - head) >> 4;
      for (int64_t i = lane; i < nvec; i += 32)
        dx_stg16(dst + head + i*16,dx_ld16_any(src + head + i*16,a.tmp_end16));
      const int64_t done = head + nvec*16;
      if ((int64_t) lane < n - done) dst[done + lane] = src[done + lane];
    }
}

}  // namespace

int dxk_qv_assemble(dx_ctx *ctx, const uint8_t *d_tmp, size_t tmp_n, const QvDecEntry *d_ent,
                    const int64_t *d_src, int64_t count, const char *d_prefix, int plen, uint8_t *d_out)
{ if (count == 0) return DX_OK;
  AsmArgs a;
  a.tmp = d_tmp; a.tmp_end16 = d_tmp + ((tmp_n + 15) & ~(size_t) 15);
  a.ent = d_ent; a.src = d_src; a.count = count; a.prefix = d_prefix; a.plen = plen; a.out = d_out;
  int64_t grid = (count + 7) / 8;
  if (grid > (int64_t) ctx->sm_count * 8) grid = (int64_t) ctx->sm_count * 8;
  DX_PROF_BEGIN(ctx); k_qv_assemble<<<(unsigned) grid,256,0,ctx->stream>>>(a);
  DX_LAUNCHED(ctx,"k_qv_assemble");
  return DX_OK;
}

int dxk_qv_decode5x(dx_ctx *ctx, const uint8_t *d_in, size_t n, const QvDecTables4 *d_tab,
                    int delchar, int subchar, int upper, int write, int64_t count,
                    const int64_t *d_start, const int32_t *d_rlen, const QvDecEntry *d_ent,
                    const char *d_prefix, int plen, uint8_t *d_out, int64_t *d_soff, int32_t *d_status,
                    const int64_t *d_limit, const int32_t *d_order, const int64_t *d_toff,
                    const int64_t *d_endat);

int dxk_qv_decode5(dx_ctx *ctx, const uint8_t *d_in, size_t n, const QvDecTables4 *d_tab,
                   int delchar, int subchar, int upper, int write, int64_t count,
                   const int64_t *d_start, const int32_t *d_rlen, const QvDecEntry *d_ent,
                   const char *d_prefix, int plen, uint8_t *d_out, int64_t *d_soff, int32_t *d_status)
{ return dxk_qv_decode5x(ctx,d_in,n,d_tab,delchar,subchar,upper,write,count,d_start,d_rlen,d_ent,d_prefix,plen,
                         d_out,d_soff,d_status,NULL,NULL,NULL,NULL);
}

int dxk_qv_decode5x(dx_ctx *ctx, const uint8_t *d_in, size_t n, const QvDecTables4 *d_tab,
                    int delchar, int subchar, int upper, int write, int64_t count,
                    const int64_t *d_start, const int32_t *d_rlen, const QvDecEntry *d_ent,
                    const char *d_prefix, int plen, uint8_t *d_out, int64_t *d_soff, int32_t *d_status,
                    const int64_t *d_limit, const int32_t *d_order, const int64_t *d_toff,
                    const int64_t *d_endat)
{ if (count == 0) return DX_OK;
  unsigned long long *d_ticket = (unsigned long long *) dx_arena_get(ctx,8);
  if (d_ticket == NULL) return DX_E_NOMEM;
  DX_CUDA(ctx,cudaMemsetAsync(d_ticket,0,8,ctx->stream));
  Dec5Args a;
  a.in = d_in; a.n = (int64_t) n; a.tab = d_tab;
  a.delchar = delchar; a.subchar = subchar; a.upper = upper; a.write = write;
  a.count = count; a.start = d_start; a.rlen = d_rlen; a.ent = d_ent;
  a.prefix = d_prefix; a.plen = plen; a.out = d_out; a.soff = d_soff; a.status = d_status;
  a.ticket = d_ticket;
  a.limit = d_limit; a.order = d_order; a.toff = d_toff; a.endat = d_endat;
  a.dbg = NULL;
  const size_t smem = sizeof(Shared5);
  DX_CUDA(ctx,cudaFuncSetAttribute(k_qv_decode5,cudaFuncAttributeMaxDynamicSharedMemorySize,(int) smem));
  int64_t grid = (count + kWarps - 1) / kWarps;
  if (grid > ctx->sm_count) grid = ctx->sm_count;
  DX_PROF_BEGIN(ctx); k_qv_decode5<<<(unsigned) grid,kThreads,smem,ctx->stream>>>(a);
  DX_LAUNCHED(ctx,write == 1 ? "k_qv_decode5" : write >= 2 ? "k_qv_decode5_spec" : "k_qv_walk5");
  return DX_OK;
}
