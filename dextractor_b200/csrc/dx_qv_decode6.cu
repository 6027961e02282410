// dx_qv_decode6.cu -- .dexqv entry decoder, one LANE per entry (the library's main decoder).
//
// Replaces Decode / Decode_Run (reference QV.c:510-691) + Packed_Length / Unpack_Tag
// (QV.c:823-847) + the per-entry text output of undexqv.c:182-207.
//
// A Huffman stream stores no code boundaries, so a stream can only be split among threads by
// speculation (dx_qv_decode5.cu: every symbol is decoded 2-3 times and a third of the lanes idle).
// But a 2 GB file holds ~40 000 independent entries: here every lane of a warp decodes ONE WHOLE
// ENTRY sequentially -- the reference's loop, one table lookup per one or two symbols, no
// speculation.  The 32 entries of a warp are neighbours in the longest-first ticket order, so their
// lengths agree within a few percent and the lanes stay busy together.  A lane is a single chain
// of dependent lookups (~50-100 cycles per lookup), so the kernel lasts as long as its longest
// entry: entries too long for that go to the warp-per-entry kernel; the host picks the cut
// (dxk_qv_decode6x, ticket_plan in dx_api.cpp).
//
// What a sequential lane needs to be fast (every item below was measured with ncu first):
//   * the five lines of an entry are five PHASES of one loop, and the warp re-joins with
//     __syncwarp at every phase boundary -- left to the compiler's reconvergence the lanes drifted
//     apart after the second line and ran alone (1.0 threads per instruction);
//   * 12-bit decode tables for all four streams in shared memory; plain streams decode two symbols
//     per lookup, run-length streams a whole (run, symbol) item per lookup;
//   * no branch inside a batch of 8 lookups: a table entry that needs anything special (escape,
//     code longer than 12 bits, long run) takes no bits and gives no symbols, so a lane that meets
//     one idles until the end of the batch, where the slow step handles it -- from shared memory
//     (one-code tables, sorted lists of the long codes), never from global memory;
//   * the bit window is 96 bits in registers (hi always full, so a refill never sits on the
//     lookup -> shift -> lookup chain), refilled without a branch every second lookup from a 16-word
//     per-lane ring in shared memory ([word][lane]: conflict free); the ring is topped up with
//     16-byte global loads issued three quads ahead; the byte misalignment of a stream is removed
//     when a quad enters the ring;
//   * output goes through a 64-byte per-lane ring in shared memory (pitch 84: lanes at the same
//     offset hit different banks) and leaves in aligned 16-byte stores; a batch writes past the
//     ring's end into 20 bytes of slack that are wrapped around once per batch.  The five lines of an
//     entry are contiguous in the text, so only the first and last block of an entry are written
//     bytewise.  Run-length streams keep the ring pre-filled with the run character: a run is an
//     addition to the write pointer.

#include <stdio.h>
#include <stdlib.h>
#include "dx_internal.h"
#include "dx_common.cuh"

namespace {

constexpr int kMaxWarps6 = 16;                  // warps per CTA: chosen per launch, <= this
constexpr int kRingW    = 16;                   // stream words per lane in the input ring
constexpr int kOutRing  = 64;                   // bytes per lane in the output ring
constexpr int kOutSlack = 20;                   // a batch of the plain loop may run this far past the ring's end
constexpr int kOutPitch = 84;                   // pitch of a lane's ring (21 words: odd, so conflict free)
constexpr int kBatch    = 8;                    // lookups between two polls of the rings
constexpr uint32_t kFastRun = 31;               // longest run the one-lookup (run, symbol) table holds

struct Dec6Args
{ const uint8_t *in;
  int64_t        n;
  const QvDecTables4 *tab;
  int32_t        delchar, subchar, upper, write;   // write: 1 text + header, 2 lines only (speculative,
                                                   //        per-entry status)
  int64_t        first, count;                     // tickets [first, count)
  const int64_t *start;        // first stream byte of each entry (after beg/end/qv)
  const int32_t *rlen;
  const QvDecEntry *ent;       // output placement (write == 1, or write == 2 with ent)
  const int64_t *toff;         // write == 2 without ent: where the entry's lines go
  const char    *prefix; int32_t plen;
  uint8_t       *out;
  int64_t       *soff;         // [count][6] or NULL
  int32_t       *status;       // [count] (write == 2) or [1] (write == 1)
  const int64_t *limit;        // per entry: first byte the entry may not reach (NULL: the image end)
  const int32_t *order;        // ticket -> entry (long entries first), NULL: identity
  const int64_t *endat;        // per entry: the byte its streams must end at (known offsets), NULL: any
};

// shared memory: the tables, then per warp an input ring and an output ring
struct Tables6
{ uint32_t tab[4][4096];       // del, ins, mrg, sub: two-symbol table or (run, symbol) table
  uint16_t one[2][2][4096];    // run-length streams (0 del, 1 sub): run codes, symbol codes (slow step)
  uint32_t longs[6][256];      // codes longer than 12 bits (QvDecTables4::longs)
  int32_t  nlong[8];
  int32_t  type[8];
};
constexpr size_t kWarpBytes6 = (size_t) kRingW*32*4 + 32*kOutPitch + 4*32*16;   // + the del-line ring of the tag phase

extern __shared__ __align__(16) uint8_t dx_dec6_smem[];

// ---- asynchronous global -> shared copies (LDGSTS): the data never passes through registers, so
//      nothing waits for it until cp_wait says so (a register pipeline of quads had the compiler
//      rotate registers with MOVs that stalled on the youngest load)
__device__ __forceinline__ void cp_async4(void *smem, const void *g, bool ok)
{ const uint32_t d = (uint32_t) __cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" :: "r"(d), "l"(g), "r"(ok ? 4 : 0) : "memory");   // 0: zero fill, nothing read
}
__device__ __forceinline__ void cp_async16_cg(void *smem, const void *g)
{ const uint32_t d = (uint32_t) __cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(d), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }

// ---- the lane's input: a bit window over a byte-aligned stream of little-endian 32-bit words ----
// The ring holds RAW aligned words of the image ([word][lane], 16 words); stream word j is
// funnel(raw[sw+j], raw[sw+j+1]) by the stream's byte skew, formed when the window is refilled.
// Quads are copied in by cp.async, one commit group each; the two youngest groups may be in flight.
struct BitIn
{ uint32_t hi;                 // the next 32 stream bits, always all valid
  uint32_t mid, lo;            // the `s` bits after them, left aligned in mid:lo (zero beyond)
  int32_t  s;                  // > 32 after every refill; a step may take up to 24
  uint32_t praw;               // raw word rd-1
  uint32_t rd, st, rd0;        // ring: next raw word to read / raw words issued / rd of the first word
  uint32_t sb8;                // byte skew of the stream against the aligned words, in bits
  const uint32_t *src, *endw;  // next raw quad to copy / first word that may not be read
  const uint32_t *safe;        // an address that may always be named (copies of size 0 past the image)
  uint32_t *ring;              // &ring[warp][0][lane]
  uint64_t base;               // address of raw word 0

  __device__ __forceinline__ void issue_quad()
  { uint32_t *r = ring + (st & (kRingW-1))*32;
    const bool ok = (src < endw);                            // quads are 16-byte aligned, endw too
    const uint32_t *q = ok ? src : safe;
    cp_async4(r,q,ok); cp_async4(r + 32,q + 1,ok); cp_async4(r + 64,q + 2,ok); cp_async4(r + 96,q + 3,ok);
    cp_commit();
    st += 4; src += 4;
  }
  // at least 5 complete words ahead of rd (the two youngest quads do not count)
  __device__ __forceinline__ void top_up()
  { while (st - rd <= 12u) issue_quad();
    cp_wait<2>();
  }
  // ... the same for the fast loops, whose batches take at most 3 words: one quad is enough
  __device__ __forceinline__ void top_up_once()
  { if (st - rd <= 12u) issue_quad();
    cp_wait<2>();
  }

  // bits consumed since the stream's first bit
  __device__ __forceinline__ uint32_t cons() const { return (rd - rd0 - 1u)*32u - 32u - (uint32_t) s; }

  __device__ __forceinline__ uint32_t next_word()
  { const uint32_t cur = ring[(rd & (kRingW-1))*32];
    const uint32_t x = __funnelshift_r(praw,cur,sb8);
    praw = cur;
    return x;
  }

  template <bool SWAP>         // SWAP: the stream is a byte string, first byte first (packed tags)
  __device__ __forceinline__ void refill()
  { if (s <= 32)
      { uint32_t x = next_word();
        if (SWAP) x = __byte_perm(x,0,0x0123);
        rd++;
        mid |= __funnelshift_rc(x,0u,(uint32_t) s);
        lo   = __funnelshift_lc(0u,x,32u - (uint32_t) s);
        s += 32;
      }
  }
  // the same without a branch (fast loops): for s > 32 both shifts clamp to "nothing"
  __device__ __forceinline__ void refill_flat()
  { const uint32_t cur = ring[(rd & (kRingW-1))*32];
    const uint32_t x = __funnelshift_r(praw,cur,sb8);
    mid |= __funnelshift_rc(x,0u,(uint32_t) s);
    lo  |= __funnelshift_lc(0u,x,(uint32_t) (32 - s));
    const bool p = (s <= 32);
    praw = p ? cur : praw;
    rd += p ? 1u : 0u;
    s  += p ? 32 : 0;
  }

  template <bool SWAP>
  __device__ __forceinline__ void init(const uint8_t *p, const uint8_t *image_end, uint32_t *ring_lane)
  { const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    cp_wait<0>();                                            // nothing of the previous stream in flight
    ring = ring_lane;
    src = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t) 15);
    endw = reinterpret_cast<const uint32_t *>((reinterpret_cast<uintptr_t>(image_end) + 15) & ~(uintptr_t) 15);
    base = (uint64_t) (a & ~(uintptr_t) 15);
    safe = reinterpret_cast<const uint32_t *>((reinterpret_cast<uintptr_t>(image_end) - 16) & ~(uintptr_t) 15);
    sb8 = (uint32_t) (a & 3) * 8u;
    rd0 = (uint32_t) (a & 15) >> 2; rd = rd0; st = 0;
    issue_quad(); issue_quad(); issue_quad(); issue_quad();
    cp_wait<2>();                                            // raw words 0..7 are there
    praw = ring[(rd & (kRingW-1))*32]; rd++;
    uint32_t w0 = next_word(); rd++;
    uint32_t w1 = next_word(); rd++;
    uint32_t w2 = next_word(); rd++;
    if (SWAP) { w0 = __byte_perm(w0,0,0x0123); w1 = __byte_perm(w1,0,0x0123); w2 = __byte_perm(w2,0,0x0123); }
    hi = w0; mid = w1; lo = w2; s = 64;
  }

  __device__ __forceinline__ void take(uint32_t len)           // len < 32, len <= s
  { hi  = __funnelshift_l(mid,hi,len);
    mid = __funnelshift_l(lo,mid,len);
    lo <<= len;
    s -= (int32_t) len;
  }

  // first byte of the image that has not been handed to the window yet
  __device__ __forceinline__ uint64_t reached() const { return base + (uint64_t) rd*4u; }
};

// the first block of an entry shares its 16 bytes with the end of the entry before it: bytes
// [head, 16) only.  Out of line (by value): once per entry, but inlined at every flush otherwise.
__device__ __noinline__ void store_head6(uint8_t *g, uint4 v, uint32_t head)
{ const uint32_t w[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
  for (int k = 0; k < 16; k++)
    if ((uint32_t) k >= head) g[k] = (uint8_t) (w[k >> 2] >> (8*(k & 3)));
}

// ---- the lane's output: bytes appended to one contiguous span of the text -------------------------
struct OutSt
{ uint8_t *gbase;              // 16-byte aligned; byte counter t <-> gbase + t
  uint32_t wr, fl, head;       // appended / flushed (multiple of 16) / bytes of block 0 that are not ours
  uint8_t *ring;               // this lane's 64 (+ slack) bytes of shared memory

  __device__ __forceinline__ void init(uint8_t *dst, uint8_t *ring_lane)
  { const uintptr_t a = reinterpret_cast<uintptr_t>(dst);
    gbase = reinterpret_cast<uint8_t *>(a & ~(uintptr_t) 15);
    head = (uint32_t) (a & 15); wr = head; fl = 0; ring = ring_lane;
  }
  __device__ __forceinline__ void put(uint32_t c) { ring[wr & (kOutRing-1)] = (uint8_t) c; wr++; }

  // one complete block, if there is one; FILL: the block is filled with the byte again (run streams)
  template <bool FILL>
  __device__ __forceinline__ void flush_one(uint32_t fill4)
  { if (wr - fl >= 16u)
      { uint32_t *b = reinterpret_cast<uint32_t *>(ring + (fl & (kOutRing-1)));
        const uint4 v = make_uint4(b[0],b[1],b[2],b[3]);
        if (fl == 0 && head != 0) store_head6(gbase,v,head);
        else                      dx_stg16(gbase + fl,v);
        if (FILL) { b[0] = fill4; b[1] = fill4; b[2] = fill4; b[3] = fill4; }
        fl += 16;
      }
  }
  template <bool FILL>
  __device__ __forceinline__ void flush(uint32_t fill4)
  { while (wr - fl >= 16u) flush_one<FILL>(fill4); }

  // every byte appended so far is in global memory afterwards; the state does not change
  __device__ __forceinline__ void sync_partial()
  { flush<false>(0);
    const uint32_t from = (fl == 0) ? head : fl;
    for (uint32_t t = from; t < wr; t++) gbase[t] = ring[t & (kOutRing-1)];
  }
  // bytes [wr, fl + 64) of the ring := c
  __device__ __forceinline__ void prefill(uint32_t c)
  { for (uint32_t t = wr; t < fl + kOutRing; t++) ring[t & (kOutRing-1)] = (uint8_t) c; }

  // append r copies of the byte the ring is pre-filled with
  __device__ __forceinline__ void skip(uint32_t r, uint32_t fill4)
  { while (true)
      { const uint32_t room = fl + 48u - wr;           // >= 33: flush leaves fewer than 16 pending
        const uint32_t a = min(r,room);
        wr += a; r -= a;
        flush<true>(fill4);
        if (r == 0) break;
      }
  }
};

// ---- slow steps: everything comes from shared memory -----------------------------------------------
// a code longer than 12 bits: sym | len << 8, or 0x100 | E6_BAD1 when no code owns the window (garbage)
#define E6_BAD   0x2000u                /* multi entries: bit 13 */
#define E6_BAD1  0x8000u                /* single entries: bit 15 */
__device__ __noinline__ uint32_t long_code6(const uint32_t *lg, int n, uint32_t w)
{ const uint32_t w16 = w >> 16;
  int lo = 0, hi = n;                                   // last entry whose code16 <= w16
  while (lo < hi)
    { const int m = (lo + hi) >> 1;
      if ((lg[m] >> 16) <= w16) lo = m + 1; else hi = m;
    }
  if (lo == 0) return 0x100u | E6_BAD1;
  const uint32_t e = lg[lo-1];
  const uint32_t len = (e >> 8) & 0xffu;
  if (((e >> 16) ^ w16) >> (16u - len)) return 0x100u | E6_BAD1;
  return e & 0xffffu;
}
// ... as an entry of the plain-stream table
__device__ __forceinline__ uint32_t long_entry6(const uint32_t *lg, int n, int type, uint32_t w)
{ const uint32_t f = long_code6(lg,n,w);
  const uint32_t len = (f >> 8) & 31u, c = f & 0xffu;
  const uint32_t bad = (f & E6_BAD1) ? E6_BAD : 0u;
  if (type == 2 && c == 255u)
    return (len + 8u) | (1u << 5) | 0x80u | (len << 8) | (255u << 16) | bad;
  return len | (1u << 5) | (len << 8) | (c << 16) | bad;
}

// multi entry (QvDecTables4): bits 0-4 total length, 5-6 symbols, 7 escape, 8-12 length of the first
// code, 16-23 / 24-31 the symbols.  In shared memory an escape entry keeps bits 7-12 only: to the
// fast loop it is "no bits, no symbols" like the empty entry of a long code.
#define E6_LEN(e)   ((e) & 31u)
#define E6_N(e)     (((e) >> 5) & 3u)
#define E6_LEN0(e)  (((e) >> 8) & 31u)

struct Lane
{ BitIn in; OutSt out;
  uint32_t bad;
  uint64_t lim;                // address the entry may not read past
};

// one symbol of a plain stream the slow way; returns the position of the last item read
__device__ __forceinline__ uint32_t plain_step(Lane &ln, const uint32_t *mt, const uint32_t *lg, int nlg, int type)
{ BitIn &in = ln.in;
  const uint32_t w = in.hi;
  uint32_t e = mt[w >> 20];
  if (e == 0u) { e = long_entry6(lg,nlg,type,w); ln.bad |= e & E6_BAD; }
  const uint32_t l0 = E6_LEN0(e);
  uint32_t c0 = (e >> 16) & 0xffu, adv = l0, last = in.cons();
  if (e & 0x80u) { c0 = (w << l0) >> 24; last += l0; adv += 8u; }
  ln.out.put(c0);
  in.take(adv);
  in.refill<false>();
  return last;
}

// one plain stream of L symbols (QV.c:510-599); returns the bytes the stream occupies in the file.
// `act`: the lanes of the warp that enter together.  Every loop head is a __ballot_sync over the
// lanes still in the loop: it is the loop condition AND the point where the lanes re-join (left to
// the compiler, lanes that finish a poll early start the next batch alone).
__device__ __forceinline__ uint32_t plain_stream(Lane &ln, uint32_t act, const uint32_t *mt, const uint32_t *lg,
                                                 int nlg, int type, uint32_t L)
{ BitIn &in = ln.in; OutSt &out = ln.out;
  uint32_t cnt = 0, last = 0;
  if (L > 0) in.top_up();
  // ---- fast: batches of kBatch lookups, up to two symbols each, no branch inside a batch ----------
  while (true)
    { const bool go = (cnt + 2u*kBatch + 2u < L);
      act = __ballot_sync(act,go);
      if (!go) break;
      const uint32_t wo = out.wr & (kOutRing-1);
      uint8_t *p = out.ring + wo;
#pragma unroll
      for (int it = 0; it < kBatch; it++)
        { const uint32_t e = mt[in.hi >> 20];
          p[0] = (uint8_t) (e >> 16);
          p[1] = (uint8_t) (e >> 24);
          p += E6_N(e);
          in.take(E6_LEN(e));
          if (it & 1) in.refill_flat();                     // two lookups take at most 24 bits
        }
      const uint32_t made = (uint32_t) (p - (out.ring + wo));
      out.wr += made; cnt += made;
      if (wo + made > (uint32_t) kOutRing)                  // ran into the slack: wrap it around
        { const uint32_t *src = reinterpret_cast<const uint32_t *>(out.ring + kOutRing);
          uint32_t *dst = reinterpret_cast<uint32_t *>(out.ring);
#pragma unroll
          for (int k = 0; k < kOutSlack/4; k++) dst[k] = src[k];
        }
      out.flush_one<false>(0);                              // 15 pending + 16 made: at most one block
      in.top_up_once();
      // an entry the fast loop cannot take under the window: symbols the slow way until it is gone
      while (E6_N(mt[in.hi >> 20]) == 0u && cnt + 2u < L)
        { plain_step(ln,mt,lg,nlg,type);
          cnt++;
          out.flush_one<false>(0);
          in.top_up();
        }
      if (in.reached() > ln.lim) { ln.bad = 1; cnt = L; last = 0; }
    }
  // ---- the last symbols one at a time: the position of the last item (the literal of an escape)
  //      fixes the stream's length in the file (QV.c:537-551)
  while (cnt < L)
    { last = plain_step(ln,mt,lg,nlg,type);
      cnt++;
      out.flush_one<false>(0);
      in.top_up_once();
    }
  return (L == 0 || ln.bad) ? 0u : ((last + 47u) >> 5) * 4u;
}

// one run-length stream (QV.c:604-691): (run of rc, one other symbol)*
// pt: the stream's (run, symbol) table -- one lookup decodes a whole item when the run is at most
// kFastRun, both codes together have at most 12 bits and nothing is escaped: bits 0-4 the item's
// length, 8-15 the run, 16-23 the symbol; 0 = everything else (slow step: rt / st, the one-code tables).
__device__ __forceinline__ uint32_t run_stream(Lane &ln, uint32_t act, const uint32_t *pt, const uint16_t *rt, const uint16_t *st,
                                               const uint32_t *lgr, int nlgr, const uint32_t *lgs, int nlgs,
                                               bool esc, uint32_t rc, uint32_t L, uint32_t *kept_out)
{ BitIn &in = ln.in; OutSt &out = ln.out;
  const uint32_t rc4 = rc * 0x01010101u;
  uint32_t cnt = 0, last = 0, kept = 0;
  *kept_out = 0;
  if (L > 0) { out.prefill(rc); in.top_up(); }
  while (true)
    { const bool go = (cnt < L);
      act = __ballot_sync(act,go);
      if (!go) break;
      // ---- fast: whole items by one lookup, while no item can reach the end of the line -----------
      if (cnt + 4u*(kFastRun + 1u) < L)
        {
#pragma unroll
          for (int it = 0; it < 4; it++)
            { const uint32_t e = pt[in.hi >> 20];
              const uint32_t r = (e >> 8) & 0xffu;
              const uint32_t adv = (e != 0u) ? r + 1u : 0u;
              if (e != 0u) out.ring[(out.wr + r) & (kOutRing-1)] = (uint8_t) (e >> 16);
              out.wr += adv; cnt += adv; kept += (e != 0u) ? 1u : 0u;
              in.take(E6_LEN(e));
              if (it & 1) in.refill_flat();
              out.flush_one<true>(rc4);                      // 15 pending + 32: at most two blocks
              out.flush_one<true>(rc4);
            }
          in.top_up_once();
          if (pt[in.hi >> 20] != 0u) continue;
        }
      // ---- one item the slow way ------------------------------------------------------------------------
      { uint32_t w = in.hi;
        uint32_t e = rt[w >> 20];
        if (e == 0u) { e = long_code6(lgr,nlgr,w); ln.bad |= e & E6_BAD1; e &= 0x1fffu; }
        uint32_t r = e & 0xffu;
        last = in.cons();
        in.take(e >> 8);
        in.refill<false>();
        if (r == 255u)
          { r = in.hi >> 16; last = in.cons();
            in.take(16);
            in.refill<false>();
          }
        if (r > L - cnt) { r = L - cnt; ln.bad = 1; }
        cnt += r;
        out.skip(r,rc4);
        if (cnt < L)
          { w = in.hi;
            e = st[w >> 20];
            if (e == 0u) { e = long_code6(lgs,nlgs,w); ln.bad |= e & E6_BAD1; e &= 0x1fffu; }
            uint32_t c = e & 0xffu;
            last = in.cons();
            in.take(e >> 8);
            in.refill<false>();
            if (esc && c == 255u)
              { c = in.hi >> 24; last = in.cons();
                in.take(8);
                in.refill<false>();
              }
            out.put(c);
            cnt++;
            kept += (c != rc);
          }
        in.top_up();
        out.flush<true>(rc4);
        if (in.reached() > ln.lim) { ln.bad = 1; cnt = L; }
      }
    }
  out.flush<true>(rc4);
  *kept_out = kept;
  return (L == 0) ? 0u : ((last + 47u) >> 5) * 4u;
}

// the tag line (Unpack_Tag, QV.c:837-847): 'n' where the deletion QV is the run character, the next
// packed tag elsewhere.  The del line is read back from global memory (the lane's own stores, through
// L2) in aligned 16-byte blocks, copied by cp.async three blocks ahead into a 4-block ring; the packed
// tags are a bit stream of their own: the (at most 16) tags of a block are taken from the window in two
// pieces.
__device__ __forceinline__ void tag_line(Lane &ln, uint32_t act, uint4 *dring, const uint8_t *del, uint32_t L,
                                         int32_t delchar, uint32_t upper)
{ BitIn &in = ln.in; OutSt &out = ln.out;
  const uint32_t caseoff = upper ? 32u : 0u;
  const uint32_t nch = 'n' - caseoff, n4 = nch * 0x01010101u;
  const uint32_t acgt = 0x74676361u - caseoff*0x01010101u;
  const uintptr_t a = reinterpret_cast<uintptr_t>(del);
  const uint4 *blk = reinterpret_cast<const uint4 *>(a & ~(uintptr_t) 15);
  int32_t p = -(int32_t) (a & 15);                    // line position of the block's first byte
  const int32_t nblk = (L > 0) ? (int32_t) (((a & 15) + L + 15) >> 4) : 0;
  if (L > 0)
    { out.prefill(nch);
      in.top_up();
      // (the packed-tag stream's quads are commit groups too: wait for ALL groups before a block
      //  is read -- the tag stream advances one word per block at most, so nothing is lost)
      if (delchar >= 0)
        for (int j = 0; j < 3; j++)
          { if (j < nblk) cp_async16_cg(dring + 32*j,blk + j);
            cp_commit();
          }
    }
  int32_t bi = 0;
  while (true)
    { const bool go = (bi < nblk);
      act = __ballot_sync(act,go);
      if (!go) break;
      const int lo = max(0,-p), hi = min(16,(int32_t) L - p);
      uint32_t m = dx_range16(lo,hi);
      if (delchar >= 0)
        { if (bi + 3 < nblk) cp_async16_cg(dring + 32*((bi + 3) & 3),blk + bi + 3);
          cp_commit();
          cp_wait<3>();                                     // block bi is there (and older tag quads)
          const uint4 v = dring[32*(bi & 3)];
          m &= ~dx_eq_mask16(v,(uint32_t) delchar);
        }
      const uint32_t k = __popc(m);
      // the block's tags: 2k <= 32 bits, in two pieces of at most 16
      const uint32_t k1 = min(k,8u), k2 = k - k1;
      uint32_t tg = 0;                                      // tag j of the block in bits 31-2j, 30-2j
      if (k1) { tg = (in.hi >> (32u - 2u*k1)) << (32u - 2u*k1); in.take(2u*k1); in.refill<true>(); }
      if (k2) { tg |= (in.hi >> (32u - 2u*k2)) << (16u - 2u*k2); in.take(2u*k2); in.refill<true>(); }
      const uint32_t w0 = out.wr - (uint32_t) lo;            // ring counter of block byte 0
      while (m)
        { const int i = __ffs(m) - 1; m &= m - 1;
          out.ring[(w0 + (uint32_t) i) & (kOutRing-1)] = (uint8_t) (acgt >> (8u*(tg >> 30)));
          tg <<= 2;
        }
      out.wr += (uint32_t) (hi - lo);
      out.flush_one<true>(n4);
      if (in.st - in.rd <= 12u) { in.issue_quad(); cp_wait<3>(); }
      p += 16; bi++;
    }
  cp_wait<0>();
  out.flush<true>(n4);
}

__device__ int fmt_int6(uint8_t *p, int32_t v)
{ char tmp[12];
  int  k = 0, len = 0;
  uint32_t u = (v < 0) ? (uint32_t) (-(int64_t) v) : (uint32_t) v;
  if (v < 0) p[len++] = '-';
  do { tmp[k++] = (char) ('0' + u % 10); u /= 10; } while (u);
  while (k) p[len++] = (uint8_t) tmp[--k];
  return len;
}

__global__ void __launch_bounds__(kMaxWarps6*32,1)
k_qv_decode6(Dec6Args a)
{ Tables6 &sm = *reinterpret_cast<Tables6 *>(dx_dec6_smem);
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, nthreads = blockDim.x;
  uint8_t *wmem = dx_dec6_smem + sizeof(Tables6) + (size_t) warp*kWarpBytes6;

  // resident tables (see plain_stream / run_stream); slot 0 del, 1 ins, 2 mrg, 3 sub
  { const QvDecTables4 *T = a.tab;
    for (int s = 0; s < 4; s++)
      { const int symtab = (s == 0) ? 0 : (s == 1) ? 2 : (s == 2) ? 3 : 4;
        const int runtab = (s == 0) ? 1 : 5;
        const int32_t rci = (s == 0) ? a.delchar : (s == 3) ? a.subchar : -1;
        if (rci >= 0)
          { const uint16_t *gr = T->single[runtab], *gs = T->single[symtab];
            const bool esc = (T->t2.type[symtab] == 2);
            uint16_t *o_r = sm.one[s == 0 ? 0 : 1][0], *o_s = sm.one[s == 0 ? 0 : 1][1];
            for (int j = threadIdx.x; j < 4096; j += nthreads)
              { const uint32_t e1 = __ldg(gr + j);
                const uint32_t r = e1 & 0xffu, l1 = e1 >> 8;
                o_r[j] = (uint16_t) e1; o_s[j] = __ldg(gs + j);
                uint32_t v = 0;
                if (e1 != 0u && r <= kFastRun && l1 < 12u)
                  { const uint32_t e2 = __ldg(gs + ((j << l1) & 0xfff));
                    const uint32_t c = e2 & 0xffu, l2 = e2 >> 8;
                    if (e2 != 0u && l1 + l2 <= 12u && !(esc && c == 255u) && c != (uint32_t) rci)
                      v = (l1 + l2) | (r << 8) | (c << 16);
                  }
                sm.tab[s][j] = v;
              }
          }
        else
          for (int j = threadIdx.x; j < 4096; j += nthreads)
            { const uint32_t e = __ldg(T->multi[symtab] + j);
              sm.tab[s][j] = (e & 0x80u) ? (e & 0x00ff1f80u) : e;
            }
      }
    for (int j = threadIdx.x; j < 6*256; j += nthreads) sm.longs[j >> 8][j & 255] = __ldg(&T->longs[j >> 8][j & 255]);
    if (threadIdx.x < 6) { sm.nlong[threadIdx.x] = T->nlong[threadIdx.x]; sm.type[threadIdx.x] = T->t2.type[threadIdx.x]; }
  }
  __syncthreads();

  // No lane leaves before the end: the lanes of a warp re-join at every phase boundary below
  // (__syncwarp over the lanes that hold a ticket).
  const int64_t t = a.first + ((int64_t) blockIdx.x*(nthreads >> 5) + warp)*32 + lane;
  const bool ticket = (t < a.count);
  const uint32_t live = __ballot_sync(DX_FULL,ticket);
  if (!ticket) return;
  const int64_t e = (a.order != NULL) ? (int64_t) a.order[t] : t;
  const int32_t Ls = a.rlen[e];
  const uint32_t L = (Ls > 0) ? (uint32_t) Ls : 0u;
  const uint8_t *image_end = a.in + a.n;
  const int64_t lim = (a.limit != NULL) ? a.limit[e] : a.n;
  Lane ln;
  ln.bad = 0;
  ln.lim = reinterpret_cast<uint64_t>(a.in) + (uint64_t) lim + 80u;
  uint32_t *ring_lane = reinterpret_cast<uint32_t *>(wmem) + lane;
  uint8_t  *line = a.out;
  bool dead = (Ls < 0);                                     // ruled out by the host, or given up
  if (!dead)
    { if (a.write == 2 && a.ent == NULL)
        line = a.out + a.toff[e];
      else
        { const QvDecEntry en = a.ent[e];
          line = a.out + en.text_off;
          if (a.write == 1)
            { uint8_t *h = a.out + en.out_off;              // "%s/%d/%d_%d RQ=0.%d\n" (undexqv.c:182)
              int hl = 0;
              for (int k = 0; k < a.plen; k++) h[hl++] = (uint8_t) a.prefix[k];
              h[hl++] = '/'; hl += fmt_int6(h+hl,en.well);
              h[hl++] = '/'; hl += fmt_int6(h+hl,en.beg);
              h[hl++] = '_'; hl += fmt_int6(h+hl,en.end);
              const char *rq = " RQ=0.";
              for (int k = 0; k < 6; k++) h[hl++] = (uint8_t) rq[k];
              hl += fmt_int6(h+hl,en.qv);
              h[hl++] = '\n';
            }
        }
    }
  ln.out.init(line,wmem + kRingW*32*4 + lane*kOutPitch);

  int64_t at = a.start[e];
  if (a.soff != NULL) a.soff[e*6] = at;
  uint32_t kept = L;
  int done = 0;                                             // phases completed
  // phases: 0 deletion QVs, 1 deletion tags, 2 insertion QVs, 3 merge QVs, 4 substitution QVs
#pragma unroll 1
  for (int ph = 0; ph < 5; ph++)
    { // who takes part in this phase is settled BEFORE the ballot: every lane of `act` then calls the
      // phase's stream function exactly once (its loop heads are ballots over these lanes)
      bool part = !dead;
      if (part && at > a.n)
        { ln.bad = 1;
          if (a.write != 1) { dead = true; part = false; } else at = a.n;
        }
      uint32_t Lp = L;
      int64_t tbytes = 0;
      if (ph == 1)
        { const uint32_t clen = (a.delchar < 0) ? L : kept;
          tbytes = (clen + 3) >> 2;
          if (at + tbytes > a.n) Lp = 0;                     // the packed tags are cut off: no tag stream
        }
      const uint32_t act = __ballot_sync(live,part);        // also where the lanes re-join
      if (!part) continue;
      if (ph == 1)
        { if (Lp > 0)
            { ln.out.sync_partial();                         // the del line is complete in global memory
              ln.in.init<true>(a.in + at,image_end,ring_lane);
            }
          tag_line(ln,act,reinterpret_cast<uint4 *>(wmem + kRingW*32*4 + 32*kOutPitch) + lane,
                   line,Lp,a.delchar,(uint32_t) a.upper);
          if (Lp != L)
            { ln.bad = 1;
              for (uint32_t k = 0; k < L; k++) { ln.out.put('n'); ln.out.flush<false>(0); }
            }
          at += tbytes;
        }
      else
        { const int slot = (ph == 0) ? 0 : ph - 1;
          const int symtab = (ph == 0) ? 0 : ph;
          const int runtab = (ph == 0) ? 1 : 5;
          const int rci = (ph == 0) ? a.delchar : (ph == 4) ? a.subchar : -1;
          uint32_t bytes;
          if (L > 0) ln.in.init<false>(a.in + at,image_end,ring_lane);
          if (rci >= 0)
            { uint32_t k2 = 0;
              const int w = (ph == 0) ? 0 : 1;
              bytes = run_stream(ln,act,sm.tab[slot],sm.one[w][0],sm.one[w][1],sm.longs[runtab],sm.nlong[runtab],
                                 sm.longs[symtab],sm.nlong[symtab],sm.type[symtab] == 2,(uint32_t) rci,L,&k2);
              if (ph == 0) kept = k2;
            }
          else
            bytes = plain_stream(ln,act,sm.tab[slot],sm.longs[symtab],sm.nlong[symtab],sm.type[symtab],L);
          at += bytes;
        }
      ln.out.put('\n');
      ln.out.flush_one<false>(0);
      if (a.soff != NULL) a.soff[e*6 + ph + 1] = at;
      done = ph + 1;
      if (ln.bad && a.write != 1) dead = true;
    }
  __syncwarp(live);
  if (Ls >= 0) ln.out.sync_partial();
  if (at > lim || Ls < 0) ln.bad = 1;
  if (a.endat != NULL && at != a.endat[e]) ln.bad = 1;     // the streams do not fill the entry
  if (a.soff != NULL)
    for (int k = done + 1; k < 6; k++) a.soff[e*6 + k] = at;
  if (a.write == 1) { if (ln.bad) atomicExch(a.status,1); }
  else a.status[e] = (ln.bad != 0);
}

}  // namespace

// Tickets [0, n_coop) -- the longest entries -- go to the warp-per-entry kernel, the rest to the
// lane-per-entry kernel.  Same contract as dxk_qv_decode5x otherwise (write = 1 or 2).
int dxk_qv_decode6x(dx_ctx *ctx, const uint8_t *d_in, size_t n, const QvDecTables4 *d_tab,
                    int delchar, int subchar, int upper, int write, int64_t count,
                    const int64_t *d_start, const int32_t *d_rlen, const QvDecEntry *d_ent,
                    const char *d_prefix, int plen, uint8_t *d_out, int64_t *d_soff, int32_t *d_status,
                    const int64_t *d_limit, const int32_t *d_order, const int64_t *d_toff, int64_t n_coop,
                    const int64_t *d_endat)
{ if (count == 0) return DX_OK;
  int rc;
  if (n_coop > count) n_coop = count;
  if (n_coop > 0 &&
      (rc = dxk_qv_decode5x(ctx,d_in,n,d_tab,delchar,subchar,upper,write,n_coop,d_start,d_rlen,d_ent,d_prefix,plen,
                            d_out,d_soff,d_status,d_limit,d_order,d_toff,d_endat)) != DX_OK) return rc;
  if (n_coop >= count) return DX_OK;
  Dec6Args a;
  a.in = d_in; a.n = (int64_t) n; a.tab = d_tab;
  a.delchar = delchar; a.subchar = subchar; a.upper = upper; a.write = write;
  a.first = n_coop; a.count = count; a.start = d_start; a.rlen = d_rlen; a.ent = d_ent;
  a.toff = d_toff; a.prefix = d_prefix; a.plen = plen; a.out = d_out; a.soff = d_soff; a.status = d_status;
  a.limit = d_limit; a.order = d_order; a.endat = d_endat;
  // one CTA per SM (the tables take 102 KB): as many warps per CTA as it takes to have every entry
  // in flight at once, up to 16; more entries than that run in waves, longest first
  const int64_t nwarps = (count - n_coop + 31) / 32;
  int64_t wpc = (nwarps + ctx->sm_count - 1) / ctx->sm_count;
  if (wpc < 1) wpc = 1;
  if (wpc > kMaxWarps6) wpc = kMaxWarps6;
  const size_t smem = sizeof(Tables6) + (size_t) wpc*kWarpBytes6;
  DX_CUDA(ctx,cudaFuncSetAttribute(k_qv_decode6,cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int) (sizeof(Tables6) + (size_t) kMaxWarps6*kWarpBytes6)));
  const int64_t grid = (nwarps + wpc - 1) / wpc;
  DX_PROF_BEGIN(ctx); k_qv_decode6<<<(unsigned) grid,(unsigned) (wpc*32),smem,ctx->stream>>>(a);
  DX_LAUNCHED(ctx,write == 1 ? "k_qv_decode6" : "k_qv_decode6_spec");
  return DX_OK;
}
