// dx_qv_stats.cu -- pass 1 of the QV coder on the device.
//
// Replaces Histogram_Seqs / Histogram_Runs (reference QV.c:702-724) and the order-dependent
// part of QVcoding_Scan (QV.c:988-1017):
//   k_find_delchar  first 'n'/'N' tag in file order -> delChar and the first entry whose
//                   deletion runs are counted (QV.c:993-1004)
//   k_probe_sub     walks entries until 100000 positions have been seen, then fixes subChar as
//                   the arg-max of the substitution histogram SO FAR (QV.c:1005-1015)
//   k_qv_hist       the four symbol histograms and the two run-length histograms, one warp per
//                   (entry, stream) line, thread-private byte counters in shared memory (plain
//                   read-modify-write, no atomics), flushed per stream with 64-bit global atomics

#include "dx_internal.h"
#include "dx_common.cuh"

namespace {


// ---- delChar ---------------------------------------------------------------------------------

__global__ void __launch_bounds__(256)
k_find_delchar(const uint8_t *text, QvEntries ent, unsigned long long *found)
{ const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarp = ((int64_t) gridDim.x * blockDim.x) >> 5;
  for (int64_t e = warp; e < ent.n; e += nwarp)
    { if ((*(volatile unsigned long long *) found >> 32) < (unsigned long long) e)
        return;                                    // an earlier entry already has one
      const int32_t rlen = ent.rlen[e];
      const uint8_t *tag = text + ent.line0[e] + (int64_t) rlen + 1;
      for (int32_t b = 0; b < rlen; b += 32)
        { int32_t k = b + lane;
          bool hit = (k < rlen) && (tag[k] == 'n' || tag[k] == 'N');
          uint32_t m = __ballot_sync(DX_FULL,hit);
          if (m)
            { if (lane == 0)
                atomicMin(found,((unsigned long long) e << 32) | (uint32_t) (b + __ffs(m) - 1));
              return;
            }
        }
    }
}

__global__ void k_pick_delchar(const uint8_t *text, QvEntries ent, const unsigned long long *found,
                               QvProbe *probe)
{ unsigned long long f = *found;
  if (f == ~0ull)
    { probe->delchar = -1; probe->e_del = ent.n; }
  else
    { int64_t e = (int64_t) (f >> 32);
      probe->delchar = text[ent.line0[e] + (uint32_t) f];
      probe->e_del   = e;
    }
}

// ---- subChar ---------------------------------------------------------------------------------

__global__ void __launch_bounds__(1024)
k_probe_sub(const uint8_t *text, QvEntries ent, uint64_t tot_in, const uint64_t *sub_in,
            QvProbe *probe)
{ __shared__ uint32_t h[256];
  __shared__ unsigned long long key[256];
  if (threadIdx.x < 256) h[threadIdx.x] = 0;
  __syncthreads();
  uint64_t tot = tot_in;
  int64_t  e = 0;
  bool     fixed = false;
  for ( ; e < ent.n; e++)
    { const int32_t rlen = ent.rlen[e];
      const uint8_t *sub = text + ent.line0[e] + 4*((int64_t) rlen + 1);
      for (int32_t k = threadIdx.x; k < rlen; k += blockDim.x)
        atomicAdd(&h[sub[k]],1u);
      tot += (uint64_t) rlen;
      if (tot >= 100000) { fixed = true; break; }
    }
  __syncthreads();
  if (threadIdx.x < 256)
    { uint64_t c = sub_in[threadIdx.x] + h[threadIdx.x];
      probe->sub_prefix[threadIdx.x] = c;
      // arg-max with the FIRST maximum winning: order by (count desc, symbol asc)
      key[threadIdx.x] = (c << 8) | (255u - threadIdx.x);
    }
  __syncthreads();
  if (threadIdx.x == 0)
    { unsigned long long best = 0;
      for (int k = 0; k < 256; k++) best = max(best,key[k]);
      probe->subchar = fixed ? (int32_t) (255u - (uint32_t) (best & 0xff)) : -1;
      probe->e_sub   = fixed ? e : ent.n;
      probe->totchar = tot;
    }
}

// ---- histograms ------------------------------------------------------------------------------
//
// Shared-memory atomics retire about two lanes per clock per SM, which made the first version of
// this kernel ATOMS-bound.  Here every THREAD owns a private set of one-byte counters in shared
// memory and increments them with plain load / add / store (no atomics, and no bank conflicts:
// counter b of thread t lives in word (b>>2)*T + t, byte b&3).  A counter that wraps to 0 adds
// 256 to a CTA-wide 64-bit histogram (one rare atomic per 256 hits).  When a warp moves on to the
// next stream (tickets are handed out in stream-major order) it sums its 32 lanes' counters with
// shuffles and adds them to the CTA-wide histogram of the stream it leaves; there is no CTA
// barrier before the end of the kernel.
//
//   RUN = false  streams without a run character: every byte is counted; the bytes of a 16-byte
//                chunk that lie outside the line are zeroed and counted in bin 0, which is
//                corrected by the (known) number of such bytes.  768 threads x 256 B.
//   RUN = true   del / sub with a run character (k_qv_hist_run): run bytes are skipped by a SWAR
//                compare (their count is recovered by subtraction on the host); the (position,
//                symbol) pairs of the other bytes are compacted into a per-warp queue and counted 32
//                at a time, together with the run length before each (position minus the queue
//                neighbour's position), from entry e_del / e_sub on.  Here the counters are one
//                32-bit histogram per WARP: __match_any groups the lanes of a batch that hit the
//                same bin and one of them adds the group's size, so no two lanes ever write the same
//                word.  4 KB per warp, 32 warps per SM.

struct HistArgs
{ const uint8_t *text;
  QvEntries      ent;
  int32_t        ns;               // streams handled by this launch
  int32_t        sidx[4];          // 0 del, 1 ins, 2 mrg, 3 sub
  int32_t        rc[4];            // run character of the stream (RUN launches)
  int64_t        efirst[4];        // first entry whose runs are counted
  unsigned long long *ticket;
  unsigned long long *ghist;       // [6][256]
  int32_t        mode;             // k_qv_hist_run: how a batch is counted (warp_count2), route hist_mode
};

constexpr int kHistQueue = 544;    // a row adds <= 512 items to < 32 left over

template <bool RUN> struct HistCfg
{ static constexpr int kThreads = RUN ? 384 : 768;
  static constexpr int kBins    = RUN ? 512 : 256;
  static constexpr int kRows    = kBins / 4;
  static constexpr int kStreams = RUN ? 2 : 4;
  static constexpr size_t kCnt  = (size_t) kRows * kThreads * 4;
  static constexpr size_t kWide = (size_t) kStreams * kBins * 8;
  static constexpr size_t kSmem = kCnt + kWide + (RUN ? (size_t) (kThreads/32) * kHistQueue * 4 : 0);
};

template <int T>
__device__ __forceinline__ void bump(uint8_t *mine, unsigned long long *wide, uint32_t b)
{ uint8_t *p = mine + (b & ~3u) * T + (b & 3u);
  const uint32_t c = (uint32_t) *p + 1u;
  *p = (uint8_t) c;
  if (c == 256u) atomicAdd(&wide[b],256ull);
}

// two counters at once: both loads are issued before either store, so the two read-modify-write
// chains overlap (the kernel is bound by that latency); a == b is folded into the second store
template <int T>
__device__ __forceinline__ void bump2(uint8_t *mine, unsigned long long *wide, uint32_t a, uint32_t b)
{ uint8_t *pa = mine + (a & ~3u) * T + (a & 3u);
  uint8_t *pb = mine + (b & ~3u) * T + (b & 3u);
  const uint32_t ca = *pa, cb = *pb;
  const uint32_t same = (a == b) ? 1u : 0u;
  const uint32_t na = ca + 1u, nb = cb + 1u + same;
  *pa = (uint8_t) na;
  *pb = (uint8_t) nb;
  if ((na == 256u && !same) || nb >= 256u)
    { if (na == 256u && !same) atomicAdd(&wide[a],256ull);
      if (nb >= 256u) atomicAdd(&wide[b],256ull);
    }
}

// the warp adds its lanes' byte counters to the CTA-wide histogram and clears them
template <bool RUN>
__device__ __noinline__ void hist_warp_flush(uint32_t *cnt, unsigned long long *wide, uint32_t pad)
{ typedef HistCfg<RUN> C;
  const int lane = threadIdx.x & 31;
  __syncwarp();
#pragma unroll 1
  for (int r = 0; r < C::kRows; r++)
    { uint32_t *w = cnt + (size_t) r * C::kThreads + threadIdx.x;
      const uint32_t v = *w;
      *w = 0;
      uint32_t a0 = v & 0x00ff00ffu, a1 = (v >> 8) & 0x00ff00ffu;     // 32 x 255 fits 16 bits
#pragma unroll
      for (int d = 16; d > 0; d >>= 1)
        { a0 += __shfl_xor_sync(DX_FULL,a0,d);
          a1 += __shfl_xor_sync(DX_FULL,a1,d);
        }
      const uint32_t mine = (lane == 0) ? (a0 & 0xffffu) : (lane == 1) ? (a1 & 0xffffu)
                          : (lane == 2) ? (a0 >> 16) : (a1 >> 16);
      if (lane < 4 && mine) atomicAdd(&wide[4*r + lane],(unsigned long long) mine);
    }
  if (lane == 0 && pad) atomicAdd(&wide[0],0ull - (unsigned long long) pad);   // bytes outside the lines
  __syncwarp();
}

template <bool RUN>
__global__ void __launch_bounds__(HistCfg<RUN>::kThreads,1)
k_qv_hist(HistArgs a)
{ typedef HistCfg<RUN> C;
  constexpr int T = C::kThreads;
  extern __shared__ __align__(16) uint8_t dx_hist_smem[];
  uint32_t *cnt = reinterpret_cast<uint32_t *>(dx_hist_smem);                  // [kRows][T] words
  unsigned long long *wide = reinterpret_cast<unsigned long long *>(dx_hist_smem + C::kCnt);
  uint32_t *queue = reinterpret_cast<uint32_t *>(dx_hist_smem + C::kCnt + C::kWide) +
                    (threadIdx.x >> 5) * kHistQueue;
  for (int i = threadIdx.x; i < C::kRows*T; i += T) cnt[i] = 0;
  for (int i = threadIdx.x; i < C::kStreams*C::kBins; i += T) wide[i] = 0;
  __syncthreads();

  const int lane = threadIdx.x & 31;
  uint8_t *mine = dx_hist_smem + 4*threadIdx.x;
  const int64_t nlines = a.ent.n;
  const int64_t total = nlines * a.ns;
  int cur = 0;
  uint32_t pad = 0;                                      // bytes counted in bin 0 that are not text
  unsigned long long next = 0;
  if (lane == 0) next = atomicAdd(a.ticket,1ull);

  while (true)
    { const int64_t u = (int64_t) __shfl_sync(DX_FULL,next,0);
      const int si = (u >= total) ? a.ns : (int) (u / nlines);
      if (si != cur)
        { hist_warp_flush<RUN>(cnt,wide + (size_t) cur*C::kBins,pad);
          pad = 0; cur = si;
        }
      if (si >= a.ns) break;
      if (lane == 0) next = atomicAdd(a.ticket,1ull);
      unsigned long long *wd = wide + (size_t) si*C::kBins;
      const int s = a.sidx[si];
      const int64_t tk = u - (int64_t) si*nlines;
      const int64_t e = (a.ent.order != NULL) ? (int64_t) a.ent.order[tk] : tk;
      const int32_t rlen = a.ent.rlen[e];
      if (rlen == 0) continue;
      const int lineidx = (s == 0) ? 0 : s + 1;                   // del | tag | ins | mrg | sub
      const uint8_t *line = a.text + a.ent.line0[e] + (int64_t) lineidx*((int64_t) rlen + 1);
      const int skew = (int) (reinterpret_cast<uintptr_t>(line) & 15);
      const uint8_t *base = line - skew;                           // 16-byte aligned
      const int32_t nchunk = (skew + rlen + 15) >> 4;
      uint4 nxt = (lane < nchunk) ? dx_ldg16(base + (int64_t) lane*16) : make_uint4(0,0,0,0);

      if (!RUN)
        { pad += (uint32_t) (nchunk*16 - rlen);
#pragma unroll 1
          for (int32_t c0 = 0; c0 < nchunk; c0 += 32)
            { const int32_t c = c0 + lane;
              uint4 v = nxt;
              nxt = (c + 32 < nchunk) ? dx_ldg16(base + (int64_t) (c + 32)*16) : make_uint4(0,0,0,0);
              if (c >= nchunk) continue;
              const int32_t p0 = c*16 - skew;                      // line position of byte 0
              if (p0 < 0 || p0 + 16 > rlen)                        // first / last chunk: zero the rest
                { const uint32_t valid = dx_range16(max(0,-p0),min(16,rlen - p0));
                  uint32_t k[4];
#pragma unroll
                  for (int q = 0; q < 4; q++)
                    { const uint32_t n4 = (valid >> (4*q)) & 15u;
                      k[q] = ((n4 & 1u) ? 0xffu : 0u) | ((n4 & 2u) ? 0xff00u : 0u) |
                             ((n4 & 4u) ? 0xff0000u : 0u) | ((n4 & 8u) ? 0xff000000u : 0u);
                    }
                  v.x &= k[0]; v.y &= k[1]; v.z &= k[2]; v.w &= k[3];
                }
              const uint32_t w[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
              for (int i = 0; i < 8; i++)                            // byte i of the low half with byte i of the high half
                bump2<T>(mine,wd,(w[i >> 2] >> ((i & 3)*8)) & 0xffu,(w[2 + (i >> 2)] >> ((i & 3)*8)) & 0xffu);
            }
        }
    }
  __syncthreads();
  for (int i = threadIdx.x; i < C::kStreams*C::kBins; i += T)
    { const unsigned long long v = wide[i];
      const int si = i / C::kBins, b = i % C::kBins;
      if (v && si < a.ns)
        { const int s = a.sidx[si];
          const int tab = (b < 256) ? s : (s == 0 ? 4 : 5);
          atomicAdd(&a.ghist[tab*256 + (b & 255)],v);
        }
    }
}

constexpr int kRunWarps   = 16;
constexpr int kRunThreads = kRunWarps * 32;
constexpr int kRunCtas    = 2;             // resident CTAs per SM (3 = 48 warps was measured: 1.19 ms against 1.01)
constexpr int kRunWarpWords = 512 + kHistQueue;          // histogram (256 symbols + 256 run lengths), queue

// the lanes < n of the warp add 1 to bin key[lane] (and, with `two`, to bin key2[lane]).
//   mode 0: every lane issues a shared-memory atomic add, equal keys are serialised by the hardware
//           (the default: 0.70 ms on the 2 GB bench file);
//   mode 1: round 1's form -- lanes with equal keys are grouped by match.any and the group's first
//           lane adds its size with a plain load / add / store (1.07 ms: the two match.any of a
//           batch, not the adds, were what the warps waited for; three CTAs per SM made it slower);
//   mode 2: match for the symbol, atomics for the run length (0.85 ms);  mode 3: the other way round
//           (0.83 ms);  mode 4 does not come here: no queue, see the kernel (0.73 ms).
// With atomics the kernel retires ~1.5 atomic lanes per clock and SM, the rate of the unit.  Counting
// the items the way k_qv_hist<plain> counts bytes -- 256 thread-private one-byte counters, no queue,
// 768 threads -- was measured too: 1.09 ms (a load / add / store chain per item inside a loop whose
// length differs from lane to lane); not kept.
__device__ __forceinline__ void warp_count2(uint32_t *hist, uint32_t key, uint32_t key2, bool two,
                                            uint32_t n, int lane, int mode)
{ const bool m1 = (mode == 1 || mode == 2), m2 = (mode == 1 || mode == 3);
  if ((uint32_t) lane < n)
    { const uint32_t mask = (n >= 32u) ? DX_FULL : ((1u << n) - 1u);
      if (m1)
        { const uint32_t peers = __match_any_sync(mask,key);
          if ((uint32_t) lane == (uint32_t) (__ffs(peers) - 1)) hist[key] += (uint32_t) __popc(peers);
        }
      else atomicAdd(&hist[key],1u);
      if (two)
        { if (m2)
            { const uint32_t peers2 = __match_any_sync(mask,key2);
              if ((uint32_t) lane == (uint32_t) (__ffs(peers2) - 1)) hist[key2] += (uint32_t) __popc(peers2);
            }
          else atomicAdd(&hist[key2],1u);
        }
    }
  __syncwarp();
}

__device__ __noinline__ void run_warp_flush(const HistArgs &a, int s, uint32_t *hist, int lane)
{ __syncwarp();
  for (int b = lane; b < 512; b += 32)
    { const uint32_t v = hist[b];
      hist[b] = 0;
      if (v)
        { const int tab = (b < 256) ? s : (s == 0 ? 4 : 5);
          atomicAdd(&a.ghist[tab*256 + (b & 255)],(unsigned long long) v);
        }
    }
  __syncwarp();
}

__global__ void __launch_bounds__(kRunThreads,kRunCtas)
k_qv_hist_run(HistArgs a)
{ extern __shared__ __align__(16) uint8_t dx_hist_smem[];
  const int lane = threadIdx.x & 31;
  uint32_t *hist  = reinterpret_cast<uint32_t *>(dx_hist_smem) + (threadIdx.x >> 5) * kRunWarpWords;
  uint32_t *queue = hist + 512;
  for (int b = lane; b < 512; b += 32) hist[b] = 0;
  __syncwarp();

  const int64_t nlines = a.ent.n;
  const int64_t total = nlines * a.ns;
  int cur = 0;
  unsigned long long next = 0;
  if (lane == 0) next = atomicAdd(a.ticket,1ull);
  while (true)
    { const int64_t u = (int64_t) __shfl_sync(DX_FULL,next,0);
      const int si = (u >= total) ? a.ns : (int) (u / nlines);
      if (si != cur)
        { run_warp_flush(a,a.sidx[cur],hist,lane);
          cur = si;
        }
      if (si >= a.ns) break;
      if (lane == 0) next = atomicAdd(a.ticket,1ull);
      const int s = a.sidx[si];
      const int64_t tk = u - (int64_t) si*nlines;
      const int64_t e = (a.ent.order != NULL) ? (int64_t) a.ent.order[tk] : tk;
      const int32_t rlen = a.ent.rlen[e];
      if (rlen == 0) continue;
      const int lineidx = (s == 0) ? 0 : s + 1;                   // del | tag | ins | mrg | sub
      const uint8_t *line = a.text + a.ent.line0[e] + (int64_t) lineidx*((int64_t) rlen + 1);
      const int skew = (int) (reinterpret_cast<uintptr_t>(line) & 15);
      const uint8_t *base = line - skew;                           // 16-byte aligned
      const int32_t nchunk = (skew + rlen + 15) >> 4;
      const uint32_t rc = (uint32_t) a.rc[si];
      const bool runs = (e >= a.efirst[si]);
      int32_t prevpos = -1;                                        // last position that is not rc
      uint32_t qn = 0;                                             // queued items (warp-uniform)
      uint4 nxt = (lane < nchunk) ? dx_ldg16(base + (int64_t) lane*16) : make_uint4(0,0,0,0);
      uint4 nx2 = (lane + 32 < nchunk) ? dx_ldg16(base + (int64_t) (lane + 32)*16) : make_uint4(0,0,0,0);
#pragma unroll 1
      for (int32_t c0 = 0; c0 < nchunk + 32; c0 += 32)            // one extra round drains the queue
        { const bool last = (c0 >= nchunk);
          if (a.mode == 4)
            { // no queue: every lane counts the items of its own chunk with shared-memory atomics; the
              // run before a lane's first item ends at the last item of the nearest lane in front of
              // it that has one (positions grow with the lane), or at the previous rounds' last item
              if (last) break;
              const int32_t c = c0 + lane;
              const uint4 v = nxt;
              nxt = nx2;
              nx2 = (c + 64 < nchunk) ? dx_ldg16(base + (int64_t) (c + 64)*16) : make_uint4(0,0,0,0);
              const int32_t p0 = c*16 - skew;
              uint32_t m = 0;
              if (c < nchunk)
                m = dx_range16(max(0,-p0),min(16,rlen - p0)) & ~dx_eq_mask16(v,rc);
              const int32_t mylast = m ? p0 + (31 - __clz(m)) : -1;
              const uint32_t has = __ballot_sync(DX_FULL,m != 0u);
              const uint32_t before = has & ((1u << lane) - 1u);
              const int32_t fromlane = __shfl_sync(DX_FULL,mylast,before ? 31 - __clz(before) : 0);
              int32_t pp = before ? fromlane : prevpos;
              while (m)
                { const int i = __ffs(m) - 1; m &= m - 1;
                  const int32_t pos = p0 + i;
                  atomicAdd(&hist[dx_byte_of(v,i)],1u);
                  if (runs) atomicAdd(&hist[256 + min(pos - pp - 1,255)],1u);
                  pp = pos;
                }
              const int32_t tail = __shfl_sync(DX_FULL,mylast,has ? 31 - __clz(has) : 0);
              if (has) prevpos = tail;
              continue;
            }
          if (!last)
            { const int32_t c = c0 + lane;
              const uint4 v = nxt;
              nxt = nx2;
              nx2 = (c + 64 < nchunk) ? dx_ldg16(base + (int64_t) (c + 64)*16) : make_uint4(0,0,0,0);
              const int32_t p0 = c*16 - skew;
              uint32_t m = 0;
              if (c < nchunk)
                m = dx_range16(max(0,-p0),min(16,rlen - p0)) & ~dx_eq_mask16(v,rc);
              const uint32_t k = __popc(m);
              const uint32_t inc = dx_warp_incl_sum(k,lane);
              uint32_t at = qn + inc - k;
              while (m)
                { const int i = __ffs(m) - 1; m &= m - 1;
                  queue[at++] = ((uint32_t) (p0 + i) << 8) | dx_byte_of(v,i);
                }
              qn += __shfl_sync(DX_FULL,inc,31);
              __syncwarp();
            }
          uint32_t done = 0;
#pragma unroll 1
          while (qn - done >= 32u || (last && done < qn))
            { const uint32_t n = min(32u,qn - done);
              uint32_t it = 0, rl = 0;
              if ((uint32_t) lane < n)
                { it = queue[done + lane];
                  const int32_t pp = (lane == 0) ? prevpos : (int32_t) (queue[done + lane - 1] >> 8);
                  rl = (uint32_t) min((int32_t) (it >> 8) - pp - 1,255);
                }
              warp_count2(hist,it & 0xffu,256u + rl,runs,n,lane,a.mode);
              prevpos = __shfl_sync(DX_FULL,(int32_t) (it >> 8),n-1);
              done += n;
            }
          // keep what is left (< 32 items) at the front of the queue
          const uint32_t left = qn - done;
          uint32_t keep = 0;
          if ((uint32_t) lane < left) keep = queue[done + lane];
          __syncwarp();
          if ((uint32_t) lane < left) queue[lane] = keep;
          qn = left;
          __syncwarp();
        }
      if (runs && prevpos < rlen-1)                                // trailing run (QV.c:713-720)
        { if (lane == 0) atomicAdd(&hist[256 + min(rlen-1-prevpos,255)],1u);
          __syncwarp();
        }
    }
}


}  // namespace

int dxk_qv_probe(dx_ctx *ctx, const uint8_t *d_text, QvEntries ent, const dx_qv_carry *carry,
                 QvProbe *h_probe)
{ QvProbe *d_probe = (QvProbe *) dx_arena_get(ctx,sizeof(QvProbe));
  unsigned long long *d_found = (unsigned long long *) dx_arena_get(ctx,8);
  uint64_t *d_sub_in = (uint64_t *) dx_arena_get(ctx,256*8);
  if (d_probe == NULL || d_found == NULL || d_sub_in == NULL) return DX_E_NOMEM;
  DX_CUDA(ctx,cudaMemsetAsync(d_probe,0,sizeof(QvProbe),ctx->stream));
  DX_CUDA(ctx,cudaMemsetAsync(d_found,0xff,8,ctx->stream));
  DX_CUDA(ctx,cudaMemcpyAsync(d_sub_in,carry->sub,256*8,cudaMemcpyHostToDevice,ctx->stream));

  const bool need_del = (carry->delchar < 0), need_sub = (carry->subchar < 0);
  if (need_del && ent.n > 0)
    { int blocks = ctx->sm_count * 4;
      DX_PROF_BEGIN(ctx); k_find_delchar<<<blocks,256,0,ctx->stream>>>(d_text,ent,d_found);
      DX_LAUNCHED(ctx,"k_find_delchar");
      DX_PROF_BEGIN(ctx); k_pick_delchar<<<1,1,0,ctx->stream>>>(d_text,ent,d_found,d_probe);
      DX_LAUNCHED(ctx,"k_pick_delchar");
    }
  if (need_sub)
    { DX_PROF_BEGIN(ctx); k_probe_sub<<<1,1024,0,ctx->stream>>>(d_text,ent,carry->totchar,d_sub_in,d_probe);
      DX_LAUNCHED(ctx,"k_probe_sub");
    }
  DX_CUDA(ctx,cudaMemcpyAsync(h_probe,d_probe,sizeof(QvProbe),cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  if (!need_del || ent.n == 0)
    { h_probe->delchar = carry->delchar; h_probe->e_del = (carry->delchar >= 0) ? 0 : ent.n; }
  if (!need_sub)
    { h_probe->subchar = carry->subchar; h_probe->e_sub = 0;
      memcpy(h_probe->sub_prefix,carry->sub,sizeof(carry->sub));
    }
  return DX_OK;
}

int dxk_qv_hist(dx_ctx *ctx, const uint8_t *d_text, QvEntries ent, const QvProbe *h_probe,
                uint64_t *h_hist, int32_t *h_newline_inside)
{ if (h_newline_inside) *h_newline_inside = 0;
  memset(h_hist,0,6*256*8);
  if (ent.n == 0) return DX_OK;
  unsigned long long *d_hist = (unsigned long long *) dx_arena_get(ctx,6*256*8 + 16);
  if (d_hist == NULL) return DX_E_NOMEM;
  DX_CUDA(ctx,cudaMemsetAsync(d_hist,0,6*256*8 + 16,ctx->stream));
  HistArgs plain, run;
  memset(&plain,0,sizeof(plain)); memset(&run,0,sizeof(run));
  plain.text = run.text = d_text; plain.ent = run.ent = ent;
  plain.ghist = run.ghist = d_hist;
  plain.ticket = d_hist + 6*256; run.ticket = d_hist + 6*256 + 1;
  run.mode = (int32_t) ctx->route[DXR_HIST_MODE];
  for (int s = 0; s < 4; s++)
    { const int32_t rc = (s == 0) ? h_probe->delchar : (s == 3) ? h_probe->subchar : -1;
      HistArgs &h = (rc >= 0) ? run : plain;
      h.sidx[h.ns] = s; h.rc[h.ns] = rc;
      h.efirst[h.ns] = (s == 0) ? h_probe->e_del : h_probe->e_sub;
      h.ns++;
    }
  // (function attributes are per device: set them on every call, a process may hold several contexts)
  DX_CUDA(ctx,cudaFuncSetAttribute(k_qv_hist<false>,cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int) HistCfg<false>::kSmem));
  DX_CUDA(ctx,cudaFuncSetAttribute(k_qv_hist_run,cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int) (kRunWarps*kRunWarpWords*4)));
  if (plain.ns > 0)
    { DX_PROF_BEGIN(ctx);
      k_qv_hist<false><<<ctx->sm_count,HistCfg<false>::kThreads,HistCfg<false>::kSmem,ctx->stream>>>(plain);
      DX_LAUNCHED(ctx,"k_qv_hist_plain");
    }
  if (run.ns > 0)
    { DX_PROF_BEGIN(ctx);
      k_qv_hist_run<<<ctx->sm_count*kRunCtas,kRunThreads,kRunWarps*kRunWarpWords*4,ctx->stream>>>(run);
      DX_LAUNCHED(ctx,"k_qv_hist_run");
    }
  DX_CUDA(ctx,cudaMemcpyAsync(h_hist,d_hist,6*256*8,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  return DX_OK;
}
