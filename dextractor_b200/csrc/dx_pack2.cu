// dx_pack2.cu -- the 2-bit codec, vectorised (the kernels dx_dexta_* / dx_undexta_* use first; the
// byte-serial kernels of dx_pack.cu remain as the path for unusual layouts).
//
// Replaces Number_Read / Number_Arrow + Compress_Read (reference DB.c:393-441, 319-338) and
// Uncompress_Read + Lower_/Upper_Read / Letter_Arrow (DB.c:342-389) with the line wrapping of
// undexta.c:263-270, for all entries of a file at once.
//
//   k_fa_measure2  one warp per entry: header fields, first sequence line -> width; the symbol count
//                  follows from the size of the entry's text and the width IF the lines form the
//                  usual lattice -- k_fa_pack2 checks that by counting what it packs
//   k_fa_pack2     one warp per entry, 16 text bytes per lane per round: SWAR compares give the 2-bit
//                  codes of all 16 bytes, a multiply gathers 4 codes into a byte, newlines are
//                  squeezed out, and the lanes' bit strings are concatenated with the shuffle-based
//                  writer of dx_bits.cuh (no shared atomics); output leaves through aligned stores
//   k_unpack2      one warp per entry, one ALIGNED 16-byte store per lane per round: the 32 bits
//                  that hold the round's 16 symbols come from two cached word loads and a funnel
//                  shift, PRMT maps four 2-bit codes to four characters at a time, and the newline of
//                  a wrapped line is spliced in with byte shifts
//   k_pk_*         per-entry planning of a decode on the device (header-line lengths and text
//                  offsets are prefix sums), so that the host only verifies the chain of entries

#include "dx_internal.h"
#include "dx_common.cuh"
#include "dx_bits.cuh"

namespace {

constexpr int kP2Warps   = 8;
constexpr int kP2Threads = kP2Warps * 32;
constexpr int kP2Stage   = 192;               // words per warp; a round adds at most 32
constexpr int kLineLimit = 99998;             // dexta.c:21,168: MAX_BUFFER-2 characters per line

// ---- codes ---------------------------------------------------------------------------------------------

// four text bytes -> their four 2-bit codes in one byte, first symbol in the top bits (DB.c:333-334)
template <int KIND>
__device__ __forceinline__ uint32_t codes4(uint32_t w)
{ uint32_t b0, b1;                             // 0x80 per byte: bit 0 / bit 1 of the code
  if (KIND == DX_FASTA)                        // DB.c:394-411: acgt / ACGT -> 0123, everything else 0
    { const uint32_t x = w | 0x20202020u;
      const uint32_t mc = dx_eq_mask(x,'c'), mg = dx_eq_mask(x,'g'), mt = dx_eq_mask(x,'t');
      b0 = mc | mt; b1 = mg | mt;
    }
  else                                         // DB.c:419-436: '1','2','3' -> 0,1,2 ; 'G' -> 2 ; else 3
    { const uint32_t m1 = dx_eq_mask(w,'1'), m2 = dx_eq_mask(w,'2');
      const uint32_t m3 = dx_eq_mask(w,'3') | dx_eq_mask(w,'G');
      b0 = ~(m1 | m3) & 0x80808080u; b1 = ~(m1 | m2) & 0x80808080u;
    }
  const uint32_t v = (b0 >> 7) | (b1 >> 6);
  return (v * 0x40100401u) >> 24;              // byte k's code lands at bits 31-2k..30-2k
}

// exact "is any of the 16 bytes a newline"
__device__ __forceinline__ bool any_newline(uint4 v)
{ const uint32_t k = 0x0a0a0a0au;
  const uint32_t a = v.x ^ k, b = v.y ^ k, c = v.z ^ k, d = v.w ^ k;
  const uint32_t z = ((a - 0x01010101u) & ~a) | ((b - 0x01010101u) & ~b) |
                     ((c - 0x01010101u) & ~c) | ((d - 0x01010101u) & ~d);
  return (z & 0x80808080u) != 0;
}

__device__ __forceinline__ bool digits2(const uint8_t *t, int64_t &p, int64_t end, int32_t &val)
{ int64_t s = p;
  uint32_t v = 0;
  while (p < end && t[p] >= '0' && t[p] <= '9' && p - s < 9)
    v = v*10 + (t[p++] - '0');
  if (p == s || (p < end && t[p] >= '0' && t[p] <= '9')) return false;
  val = (int32_t) v;
  return true;
}

// canonical two-decimal SNR "d+.dd" -> the uint16 the reference stores (dexar.c:152-163)
__device__ __forceinline__ bool snr_field2(const uint8_t *t, int64_t &p, int64_t end, uint32_t &cnr)
{ int32_t ip = 0;
  if (!digits2(t,p,end,ip) || ip > 99999) return false;
  if (p + 3 > end || t[p] != '.' || t[p+1] < '0' || t[p+1] > '9' || t[p+2] < '0' || t[p+2] > '9')
    return false;
  const int32_t k = ip*100 + (t[p+1]-'0')*10 + (t[p+2]-'0');
  p += 3;
  if (p < end && ((t[p] >= '0' && t[p] <= '9') || t[p] == 'e' || t[p] == 'E'))
    return false;                                                    // more decimals or an exponent: host path
  const float f = (float) ((double) k / 100.0);                      // what %f into a float yields
  cnr = (f > 99.99) ? 9999u : (uint32_t) ((double) f * 100.);
  cnr &= 0xffffu;
  return true;
}

// header fields after the first '/' (dexta.c:146-157, dexar.c:146-163).  false -> host sscanf
__device__ bool parse_header2(int kind, const uint8_t *t, int64_t p, int64_t end,
                              int32_t &well, int32_t &beg, int32_t &en, int32_t aux[2])
{ p += 1;
  while (p < end && t[p] != '/') p++;
  if (p >= end) return false;
  p++;
  if (!digits2(t,p,end,well) || p >= end || t[p] != '/') return false;
  p++;
  if (!digits2(t,p,end,beg) || p >= end || t[p] != '_') return false;
  p++;
  if (!digits2(t,p,end,en)) return false;
  if (kind == DX_FASTA)
    { aux[0] = aux[1] = 0;
      if (p == end) return true;                                     // no RQ field: qv = 0
      if (p + 6 > end || t[p] != ' ' || t[p+1] != 'R' || t[p+2] != 'Q' || t[p+3] != '=' ||
          t[p+4] != '0' || t[p+5] != '.') return false;
      p += 6;
      return digits2(t,p,end,aux[0]);
    }
  if (p + 4 > end || t[p] != ' ' || t[p+1] != 'S' || t[p+2] != 'N' || t[p+3] != '=') return false;
  p += 4;
  uint32_t c[4];
  for (int k = 0; k < 4; k++)
    { if (!snr_field2(t,p,end,c[k])) return false;
      if (k < 3) { if (p >= end || t[p] != ',') return false; p++; }
    }
  aux[0] = (int32_t) (c[0] | (c[1] << 16));
  aux[1] = (int32_t) (c[2] | (c[3] << 16));
  return true;
}

// ---- measure ---------------------------------------------------------------------------------------------
// flag bits: 1 header needs the host's sscanf, 2 pack this entry symbol by symbol, 4 line too long /
// unterminated, 8 symbol count assumed from the line lattice (verified by the packer)
__global__ void __launch_bounds__(kP2Threads)
k_fa_measure2(int kind, const uint8_t *text, int64_t n, const int64_t *hdr, FaEntries ent, int32_t *anyflag)
{ // one THREAD per entry: the work is two short byte scans (header line, first sequence line) and
  // the header parse, all sequential
  const int64_t e = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= ent.n) return;
  const int64_t h0 = hdr[e];
  const int64_t stop = (e+1 < ent.n) ? hdr[e+1] : n;
  int32_t flag = 0;
  int64_t h1 = h0;                                                 // end of the header line
  while (h1 < stop && text[h1] != '\n' && h1 - h0 <= kLineLimit) h1++;
  if (h1 >= stop) { h1 = stop - 1; flag |= 4; }                   // unterminated header line
  else if (text[h1] != '\n') flag |= 4;                           // too long
  const int64_t seq = h1 + 1, region = stop - seq;
  int64_t W = 0;                                                   // length of the first sequence line
  while (seq + W < stop && text[seq + W] != '\n' && W <= kLineLimit) W++;
  if (region > 0 && text[stop-1] != '\n') flag |= 4;              // last line unterminated
  if (W > kLineLimit) flag |= 4;
  int64_t rlen = 0;
  if (region > 0 && !(flag & 4))
    { const int64_t k = region / (W + 1), rem = region % (W + 1);
      if (W >= 1 && rem != 1)
        { rlen = k*W + (rem ? rem - 1 : 0); flag |= 8; }
      else
        { for (int64_t b = seq; b < stop; b++) rlen += (text[b] != '\n'); }   // blank lines (rare)
    }
  if (rlen >= (int64_t) 1 << 30 || region >= (int64_t) 1 << 31) flag |= 4;
  int32_t well = 0, beg = 0, en = 0, aux[2] = { 0, 0 };
  if (text[h0] != '>' || !parse_header2(kind,text,h0,h1,well,beg,en,aux)) flag |= 1;
  ent.hdr[e] = h0; ent.seq[e] = seq; ent.region[e] = region;
  ent.rlen[e] = (int32_t) rlen; ent.width[e] = (int32_t) min(W,(int64_t) 0x7fffffff);
  ent.well[e] = well; ent.beg[e] = beg; ent.end[e] = en;
  ent.aux[2*e] = aux[0]; ent.aux[2*e+1] = aux[1];
  ent.flag[e] = flag;
  if (flag & 5) atomicOr(anyflag,flag & 5);
}

// ---- pack ----------------------------------------------------------------------------------------------------

struct Pack2Args
{ const uint8_t *text;
  FaEntries ent;
  int32_t lwell_in;
  uint8_t *out;
  int32_t *err;                 // set to 1 when an entry's symbol count is not the measured one
  unsigned long long *ticket;
  int32_t only_leftover;        // 1: only the entries k_fa_pack3 (dx_pack3.cu) left aside
};

template <int KIND>
__global__ void __launch_bounds__(kP2Threads)
k_fa_pack2(Pack2Args a)
{ __shared__ uint32_t stage_all[kP2Warps][kP2Stage + 4];
  const int lane = threadIdx.x & 31;
  uint32_t *stage = stage_all[threadIdx.x >> 5];
  const uint32_t fields = (KIND == DX_FASTA) ? 12u : 16u;
  unsigned long long next = 0;
  if (lane == 0) next = atomicAdd(a.ticket,1ull);
  while (true)
    { const int64_t e = (int64_t) __shfl_sync(DX_FULL,next,0);
      if (e >= a.ent.n) break;
      if (lane == 0) next = atomicAdd(a.ticket,1ull);
      const int32_t rlen = a.ent.rlen[e];
      if (a.only_leftover && !(rlen > 0 && (!(a.ent.flag[e] & 8) || a.ent.width[e] < 32))) continue;
      uint8_t *dst = a.out + a.ent.off[e];
      if (lane == 0)
        { // entry header: well-delta bytes, beg, end, qv | 4 x uint16 SNR (dexta.c:187-198)
          int32_t lwell = (e == 0) ? a.lwell_in : a.ent.well[e-1];
          const int32_t well = a.ent.well[e];
          uint8_t *h = dst;
          while (well - lwell >= 255) { *h++ = 0xff; lwell += 255; }
          *h++ = (uint8_t) (well - lwell);
          const uint32_t f[4] = { (uint32_t) a.ent.beg[e], (uint32_t) a.ent.end[e],
                                  (uint32_t) a.ent.aux[2*e], (uint32_t) a.ent.aux[2*e+1] };
          for (uint32_t k = 0; k < fields; k++)
            *h++ = (uint8_t) (f[k >> 2] >> (8*(k & 3)));
        }
      const uint32_t clen = ((uint32_t) rlen + 3u) >> 2;
      uint8_t *pay = dst + (a.ent.bytes[e] - clen);
      const uint8_t *seq = a.text + a.ent.seq[e];
      LineWalk lw; lw.set(seq,(int32_t) a.ent.region[e]);
      WarpBits wb; wb.init(stage,pay,kP2Stage);
      bool bad = false;
      int32_t last_nl = -1;                                          // region offset of the last newline
      bool toolong = false;                                          // a line of more than kLineLimit characters
      uint4 nxt = (lane < lw.nchunk) ? dx_ldg16(lw.base + (int64_t) lane*16) : make_uint4(0,0,0,0);
#pragma unroll 1
      for (int32_t c0 = 0; c0 < lw.nchunk; c0 += 32)
        { const int32_t c = c0 + lane;
          const uint4 v = nxt;
          nxt = (c + 32 < lw.nchunk) ? dx_ldg16(lw.base + (int64_t) (c + 32)*16) : make_uint4(0,0,0,0);
          const uint32_t valid = lw.valid(c);
          uint32_t nl = 0;
          if (valid && any_newline(v)) nl = dx_eq_mask16(v,'\n') & valid;
          // dexta.c:168-172: every line the reference reads has at most MAX_BUFFER-2 characters.  Gaps
          // inside a round are shorter than 512; what can be too long is the gap to the last newline
          // of an earlier round.
          { const uint32_t any = __ballot_sync(DX_FULL,nl != 0);
            if (any)
              { const int f = __ffs(any) - 1, l = 31 - __clz(any);
                const int32_t mine_first = c*16 - lw.skew + (__ffs(nl) - 1);
                const int32_t mine_last  = c*16 - lw.skew + (31 - __clz(nl));
                const int32_t first = __shfl_sync(DX_FULL,mine_first,f);
                if (first - last_nl - 1 > kLineLimit) toolong = true;
                last_nl = __shfl_sync(DX_FULL,mine_last,l);
              }
          }
          const uint32_t keep = valid & ~nl;
          const uint32_t cnt = __popc(keep);
          const uint32_t x = (codes4<KIND>(v.x) << 24) | (codes4<KIND>(v.y) << 16) |
                             (codes4<KIND>(v.z) << 8) | codes4<KIND>(v.w);
          uint32_t val = x;
          if (keep != 0xffffu)
            { val = 0;
              if (cnt)
                { const int lo = __ffs(valid) - 1, hi = 32 - __clz(valid);          // valid = [lo, hi)
                  if (nl == 0)
                    val = (x << (2*lo)) >> (32 - 2*cnt);
                  else if ((nl & (nl - 1)) == 0)                                     // one newline inside
                    { const int j = __ffs(nl) - 1;
                      const int nh = j - lo, nw = hi - j - 1;
                      const uint32_t h = nh ? (x << (2*lo)) >> (32 - 2*nh) : 0u;
                      const uint32_t l = nw ? (x << (2*(j+1))) >> (32 - 2*nw) : 0u;
                      val = (h << (2*nw)) | l;
                    }
                  else
                    { uint32_t m = keep;
                      while (m)
                        { const int i = __ffs(m) - 1; m &= m - 1;
                          val = (val << 2) | ((x >> (30 - 2*i)) & 3u);
                        }
                    }
                }
            }
          const uint32_t inc = dx_warp_incl_sum(cnt,lane);
          wb.reserve<true>(__shfl_sync(DX_FULL,inc,31)*2u,lane);
          LaneSink sk;
          sk.start(wb.bitpos() + (inc - cnt)*2u);
          sk.put(wb.stage,val,cnt*2u);
          sk.finish(wb,lane);
          if ((wb.flushed + wb.nst)*4u > clen) { bad = true; break; }   // more symbols than measured
        }
      __syncwarp();
      const uint32_t kept = wb.total() >> 1;
      if (toolong || (int32_t) a.ent.region[e] - last_nl - 1 > kLineLimit)
        { if (lane == 0) atomicMax(a.err,2); }                      // a line the reference refuses
      else if (bad || kept != (uint32_t) rlen)
        { if (lane == 0) atomicMax(a.err,1); }                      // the measured count was wrong: redo
      else
        { if (lane == 0 && wb.cbits) stage[wb.nst] = wb.carry;
          __syncwarp();
          copy_out<true>(pay + (size_t) wb.flushed*4u,stage,clen - wb.flushed*4u,lane);
        }
      __syncwarp();
    }
}

// ---- unpack --------------------------------------------------------------------------------------------------

__device__ int fmt_int2(uint8_t *p, int32_t v)
{ char tmp[12];
  int  k = 0, len = 0;
  uint32_t u = (v < 0) ? (uint32_t) (-(int64_t) v) : (uint32_t) v;
  if (v < 0) p[len++] = '-';
  do { tmp[k++] = (char) ('0' + u % 10); u /= 10; } while (u);
  while (k) p[len++] = (uint8_t) tmp[--k];
  return len;
}

struct Unpack2Args
{ int kind, upper, width;
  const uint8_t *in; const uint8_t *in_end4;         // first 4-byte aligned address past the readable image
  const PkDecEntry *ent; int64_t count;
  const char *prefix; int plen;
  uint8_t *out;
  unsigned long long *ticket;
};

__global__ void __launch_bounds__(kP2Threads)
k_unpack2(Unpack2Args a)
{ const int lane = threadIdx.x & 31;
  const uint32_t alpha = (a.kind == DX_ARROW) ? 0x34333231u          // "1234"
                        : a.upper ? 0x54474341u : 0x74676361u;       // "ACGT" / "acgt"
  const uint32_t W = (uint32_t) a.width, Wp1 = W + 1u;
  unsigned long long next = 0;
  if (lane == 0) next = atomicAdd(a.ticket,1ull);
  while (true)
    { const int64_t e = (int64_t) __shfl_sync(DX_FULL,next,0);
      if (e >= a.count) break;
      if (lane == 0) next = atomicAdd(a.ticket,1ull);
      const PkDecEntry en = a.ent[e];
      const int64_t rlen = (int64_t) en.end - en.beg;
      if (lane == 0)
        { // "%s/%d/%d_%d RQ=0.%d\n" (undexta.c:242) or " SN=%.2f,%.2f,%.2f,%.2f\n" (undexar.c:202)
          uint8_t *h = a.out + en.out_off;
          int hl = 0;
          for (int k = 0; k < a.plen; k++) h[hl++] = (uint8_t) a.prefix[k];
          h[hl++] = '/'; hl += fmt_int2(h+hl,en.well);
          h[hl++] = '/'; hl += fmt_int2(h+hl,en.beg);
          h[hl++] = '_'; hl += fmt_int2(h+hl,en.end);
          if (a.kind == DX_FASTA)
            { const char *rq = " RQ=0.";
              for (int k = 0; k < 6; k++) h[hl++] = (uint8_t) rq[k];
              hl += fmt_int2(h+hl,en.aux[0]);
            }
          else
            { const char *sn = " SN=";
              for (int k = 0; k < 4; k++) h[hl++] = (uint8_t) sn[k];
              for (int k = 0; k < 4; k++)
                { const uint32_t c = ((uint32_t) en.aux[k >> 1] >> (16*(k & 1))) & 0xffffu;
                  hl += fmt_int2(h+hl,(int32_t) (c / 100u));
                  h[hl++] = '.';
                  h[hl++] = (uint8_t) ('0' + (c % 100u) / 10u);
                  h[hl++] = (uint8_t) ('0' + c % 10u);
                  if (k < 3) h[hl++] = ',';
                }
            }
          h[hl++] = '\n';
        }
      if (rlen <= 0) continue;
      // text of the entry: rlen symbols, a '\n' after every W of them and after the last
      const int64_t tlen = rlen + (rlen + W - 1) / W;
      const uint8_t *pay = a.in + en.bin_off;
      uint8_t *dst = a.out + en.text_off;
      const int skew = (int) (reinterpret_cast<uintptr_t>(dst) & 15);
      uint8_t *base = dst - skew;                                    // 16-byte aligned
      const int64_t nchunk = (skew + tlen + 15) >> 4;
#pragma unroll 1
      for (int64_t c = lane; c < nchunk; c += 32)
        { const int64_t t0 = c*16 - skew;                            // text offset of the chunk's byte 0
          if (t0 >= 0 && t0 + 16 < tlen)
            { // interior chunk: 16 characters, at most one of them the newline of a full line
              const uint32_t line = (uint32_t) t0 / Wp1, col = (uint32_t) t0 - line*Wp1;     // tlen < 2^32
              const int64_t b = (int64_t) line*W + col;              // first symbol of the chunk
              const uint8_t *p = pay + (b >> 2);
              const uintptr_t A = reinterpret_cast<uintptr_t>(p);
              const uint32_t *a4 = reinterpret_cast<const uint32_t *>(A & ~(uintptr_t) 3);
              const uint32_t w0 = __ldg(a4);
              const uint32_t w1 = (reinterpret_cast<const uint8_t *>(a4 + 1) < a.in_end4) ? __ldg(a4 + 1) : 0u;
              const uint32_t sh = (uint32_t) (A & 3)*8u + (uint32_t) (b & 3)*2u;
              const uint32_t x = __funnelshift_l(__byte_perm(w1,0,0x0123),__byte_perm(w0,0,0x0123),sh);
              uint32_t o[4];
#pragma unroll
              for (int k = 0; k < 4; k++)
                { const uint32_t q = x >> (24 - 8*k);
                  const uint32_t sel = ((q >> 6) & 3u) | (((q >> 4) & 3u) << 4) | (((q >> 2) & 3u) << 8) | ((q & 3u) << 12);
                  o[k] = __byte_perm(alpha,0,sel);
                }
              const uint32_t j = W - col;                            // chunk position of the newline
              if (j < 16u)
                { const uint32_t s[4] = { o[0] << 8, __funnelshift_l(o[0],o[1],8), __funnelshift_l(o[1],o[2],8),
                                          __funnelshift_l(o[2],o[3],8) };
                  const uint32_t jw = j >> 2, jb = (j & 3u)*8u;
                  const uint32_t lowm = (1u << jb) - 1u;               // bytes before the newline in its word
                  const uint32_t highm = (jb == 24u) ? 0u : ~((1u << (jb + 8u)) - 1u);
#pragma unroll
                  for (int k = 0; k < 4; k++)
                    { if ((uint32_t) k > jw) o[k] = s[k];
                      else if ((uint32_t) k == jw) o[k] = (o[k] & lowm) | (0x0au << jb) | (s[k] & highm);
                    }
                }
              dx_stg16(base + c*16,make_uint4(o[0],o[1],o[2],o[3]));
            }
          else
            { // first / last chunk of the entry: byte by byte
              const int lo = (int) max((int64_t) 0,-t0), hi = (int) min((int64_t) 16,tlen - t0);
              for (int k = lo; k < hi; k++)
                { const int64_t t = t0 + k;
                  const uint64_t line = (uint64_t) t / Wp1, col = (uint64_t) t % Wp1;
                  uint32_t ch = '\n';
                  if (col != W && t != tlen - 1)
                    { const int64_t b = (int64_t) (line*W + col);
                      const uint32_t byte = pay[b >> 2];
                      ch = (alpha >> (8*((byte >> (6 - 2*(b & 3))) & 3u))) & 0xffu;
                    }
                  base[c*16 + k] = (uint8_t) ch;
                }
            }
        }
    }
}

// ---- batched in-memory reads (the Dazzler DB loader / writer form, no line structure) -----------------------
// read r: ASCII at src + src_off[r], len[r] symbols  <->  2-bit payload at dst + dst_off[r]
struct Reads2Args
{ int kind, upper;
  const uint8_t *src; const uint8_t *src_end4; const int64_t *src_off; const int32_t *len; int64_t nreads;
  uint8_t *dst; const int64_t *dst_off;
  unsigned long long *ticket;
};

template <int KIND>
__global__ void __launch_bounds__(kP2Threads)
k_compress_reads2(Reads2Args a)
{ __shared__ uint32_t stage_all[kP2Warps][kP2Stage + 4];
  const int lane = threadIdx.x & 31;
  uint32_t *stage = stage_all[threadIdx.x >> 5];
  unsigned long long next = 0;
  if (lane == 0) next = atomicAdd(a.ticket,1ull);
  while (true)
    { const int64_t r = (int64_t) __shfl_sync(DX_FULL,next,0);
      if (r >= a.nreads) break;
      if (lane == 0) next = atomicAdd(a.ticket,1ull);
      const int32_t rlen = a.len[r];
      if (rlen <= 0) continue;
      const uint32_t clen = ((uint32_t) rlen + 3u) >> 2;
      uint8_t *pay = a.dst + a.dst_off[r];
      LineWalk lw; lw.set(a.src + a.src_off[r],rlen);
      WarpBits wb; wb.init(stage,pay,kP2Stage);
      uint4 nxt = (lane < lw.nchunk) ? dx_ldg16(lw.base + (int64_t) lane*16) : make_uint4(0,0,0,0);
#pragma unroll 1
      for (int32_t c0 = 0; c0 < lw.nchunk; c0 += 32)
        { const int32_t c = c0 + lane;
          const uint4 v = nxt;
          nxt = (c + 32 < lw.nchunk) ? dx_ldg16(lw.base + (int64_t) (c + 32)*16) : make_uint4(0,0,0,0);
          const uint32_t valid = lw.valid(c);
          const uint32_t cnt = __popc(valid);
          uint32_t val = (codes4<KIND>(v.x) << 24) | (codes4<KIND>(v.y) << 16) |
                         (codes4<KIND>(v.z) << 8) | codes4<KIND>(v.w);
          if (valid != 0xffffu)
            val = cnt ? (val << (2*(__ffs(valid) - 1))) >> (32 - 2*cnt) : 0u;
          const uint32_t inc = dx_warp_incl_sum(cnt,lane);
          wb.reserve<true>(__shfl_sync(DX_FULL,inc,31)*2u,lane);
          LaneSink sk;
          sk.start(wb.bitpos() + (inc - cnt)*2u);
          sk.put(wb.stage,val,cnt*2u);
          sk.finish(wb,lane);
        }
      __syncwarp();
      if (lane == 0 && wb.cbits) stage[wb.nst] = wb.carry;
      __syncwarp();
      copy_out<true>(pay + (size_t) wb.flushed*4u,stage,clen - wb.flushed*4u,lane);
      __syncwarp();
    }
}

__global__ void __launch_bounds__(kP2Threads)
k_uncompress_reads2(Reads2Args a)
{ const int lane = threadIdx.x & 31;
  const uint32_t alpha = (a.kind == DX_ARROW) ? 0x34333231u : a.upper ? 0x54474341u : 0x74676361u;
  unsigned long long next = 0;
  if (lane == 0) next = atomicAdd(a.ticket,1ull);
  while (true)
    { const int64_t r = (int64_t) __shfl_sync(DX_FULL,next,0);
      if (r >= a.nreads) break;
      if (lane == 0) next = atomicAdd(a.ticket,1ull);
      const int64_t rlen = a.len[r];
      if (rlen <= 0) continue;
      const uint8_t *pay = a.src + a.src_off[r];
      // whole 32-bit words are loaded: the word holding the last payload byte is the last readable one
      const uint8_t *end4 = reinterpret_cast<const uint8_t *>(
                              (reinterpret_cast<uintptr_t>(pay + ((rlen + 3) >> 2)) + 3) & ~(uintptr_t) 3);
      uint8_t *dst = a.dst + a.dst_off[r];
      const int skew = (int) (reinterpret_cast<uintptr_t>(dst) & 15);
      uint8_t *base = dst - skew;                                    // 16-byte aligned
      const int64_t nchunk = (skew + rlen + 15) >> 4;
#pragma unroll 1
      for (int64_t c = lane; c < nchunk; c += 32)
        { const int64_t t0 = c*16 - skew;                            // symbol index of the chunk's byte 0
          if (t0 >= 0 && t0 + 16 <= rlen)
            { const uint8_t *p = pay + (t0 >> 2);
              const uintptr_t A = reinterpret_cast<uintptr_t>(p);
              const uint32_t *a4 = reinterpret_cast<const uint32_t *>(A & ~(uintptr_t) 3);
              const uint32_t w0 = __ldg(a4);
              const uint32_t w1 = (reinterpret_cast<const uint8_t *>(a4 + 1) < end4) ? __ldg(a4 + 1) : 0u;
              const uint32_t sh = (uint32_t) (A & 3)*8u + (uint32_t) (t0 & 3)*2u;
              const uint32_t x = __funnelshift_l(__byte_perm(w1,0,0x0123),__byte_perm(w0,0,0x0123),sh);
              uint32_t o[4];
#pragma unroll
              for (int k = 0; k < 4; k++)
                { const uint32_t q = x >> (24 - 8*k);
                  const uint32_t sel = ((q >> 6) & 3u) | (((q >> 4) & 3u) << 4) | (((q >> 2) & 3u) << 8) | ((q & 3u) << 12);
                  o[k] = __byte_perm(alpha,0,sel);
                }
              dx_stg16(base + c*16,make_uint4(o[0],o[1],o[2],o[3]));
            }
          else
            { const int lo = (int) max((int64_t) 0,-t0), hi = (int) min((int64_t) 16,rlen - t0);
              for (int k = lo; k < hi; k++)
                { const int64_t b = t0 + k;
                  const uint32_t byte = pay[b >> 2];
                  base[c*16 + k] = (uint8_t) ((alpha >> (8*((byte >> (6 - 2*(b & 3))) & 3u))) & 0xffu);
                }
            }
        }
    }
}

// ---- planning a decode on the device ----------------------------------------------------------------------------

__device__ __forceinline__ int32_t ld32(const uint8_t *p)
{ return (int32_t) ((uint32_t) p[0] | ((uint32_t) p[1] << 8) | ((uint32_t) p[2] << 16) | ((uint32_t) p[3] << 24)); }

__device__ __forceinline__ uint32_t ndig2(int32_t v)
{ uint32_t n = (v < 0);
  const uint32_t u = (v < 0) ? (uint32_t) (-(int64_t) v) : (uint32_t) v;
  n += (u >= 1000000000u) ? 10u : (u >= 100000000u) ? 9u : (u >= 10000000u) ? 8u : (u >= 1000000u) ? 7u
     : (u >= 100000u) ? 6u : (u >= 10000u) ? 5u : (u >= 1000u) ? 4u : (u >= 100u) ? 3u : (u >= 10u) ? 2u : 1u;
  return n;
}

// candidates of a .dexta/.dexar image: where the entry would end, and what the chain needs to know
// about the bytes before its fields
__global__ void k_pk_cand_prep(const uint8_t *in, int64_t n, int64_t first, int fieldbytes, const int64_t *q,
                               int64_t count, int64_t *end, int32_t *ffrun, uint8_t *last)
{ const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const int64_t qi = q[i];
  const int64_t rl = (int64_t) ld32(in + qi + 4) - ld32(in + qi);
  const int64_t stop = qi + fieldbytes + ((rl + 3) >> 2);
  end[i] = (rl < 0 || stop > n) ? -1 : stop;
  const int64_t p = qi - 1;
  if (p < first) { ffrun[i] = -1; last[i] = 0; }
  else
    { last[i] = in[p];
      int32_t r = 0;
      int64_t k = p - 1;
      while (k >= first && in[k] == 0xff && r < (1 << 20)) { r++; k--; }
      ffrun[i] = r;
    }
}

// accepted entries: bytes of header line + wrapped sequence
__global__ void k_pk_text_len(int kind, const uint8_t *in, const int64_t *q, const int32_t *cand, const int32_t *well,
                              int64_t count, int plen, int width, uint32_t *len)
{ const int64_t m = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= count) return;
  const uint8_t *f = in + q[cand[m]];
  const int32_t beg = ld32(f), en = ld32(f+4);
  uint32_t hl = (uint32_t) plen + 1u + ndig2(well[m]) + 1u + ndig2(beg) + 1u + ndig2(en);
  if (kind == DX_FASTA) hl += 6u + ndig2(ld32(f+8)) + 1u;
  else
    { hl += 4u;
      for (int k = 0; k < 4; k++)
        { const uint32_t c = (uint32_t) f[8+2*k] | ((uint32_t) f[9+2*k] << 8);
          hl += ndig2((int32_t) (c / 100u)) + 3u + (k < 3 ? 1u : 0u);
        }
      hl += 1u;
    }
  const int64_t rl = (int64_t) en - beg;
  len[m] = hl + (rl > 0 ? (uint32_t) (rl + (rl + width - 1) / width) : 0u);
}

__global__ void k_pk_build_ent(int kind, const uint8_t *in, const int64_t *q, const int32_t *cand, const int32_t *well,
                               int64_t count, int fieldbytes, int width, const int64_t *opre, const uint32_t *len,
                               PkDecEntry *ent)
{ const int64_t m = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= count) return;
  const int64_t qi = q[cand[m]];
  const uint8_t *f = in + qi;
  PkDecEntry d;
  d.well = well[m]; d.beg = ld32(f); d.end = ld32(f+4);
  d.aux[0] = ld32(f+8);
  d.aux[1] = (kind == DX_ARROW) ? ld32(f+12) : 0;
  d.bin_off = qi + fieldbytes;
  d.out_off = opre[m];
  const int64_t rl = (int64_t) d.end - d.beg;
  d.text_off = opre[m] + (int64_t) len[m] - (rl > 0 ? rl + (rl + width - 1) / width : 0);
  ent[m] = d;
}

}  // namespace

int dxk_fa_measure2(dx_ctx *ctx, int kind, const uint8_t *d_text, size_t n, const int64_t *d_hdr,
                    FaEntries ent, int32_t *d_anyflag)
{ if (ent.n == 0) return DX_OK;
  const int64_t grid = (ent.n + kP2Threads - 1) / kP2Threads;
  DX_PROF_BEGIN(ctx);
  k_fa_measure2<<<(unsigned) grid,kP2Threads,0,ctx->stream>>>(kind,d_text,(int64_t) n,d_hdr,ent,d_anyflag);
  DX_LAUNCHED(ctx,"k_fa_measure2");
  return DX_OK;
}

int dxk_fa_pack2(dx_ctx *ctx, int kind, const uint8_t *d_text, FaEntries ent, int32_t lwell_in, uint8_t *d_out,
                 int32_t *d_err, unsigned long long *d_ticket, int only_leftover)
{ if (ent.n == 0) return DX_OK;
  Pack2Args a;
  a.text = d_text; a.ent = ent; a.lwell_in = lwell_in; a.out = d_out; a.err = d_err; a.ticket = d_ticket;
  a.only_leftover = only_leftover;
  int64_t grid = (ent.n + kP2Warps - 1) / kP2Warps;
  if (grid > (int64_t) ctx->sm_count * 8) grid = (int64_t) ctx->sm_count * 8;
  DX_PROF_BEGIN(ctx);
  if (kind == DX_FASTA) k_fa_pack2<DX_FASTA><<<(unsigned) grid,kP2Threads,0,ctx->stream>>>(a);
  else                  k_fa_pack2<DX_ARROW><<<(unsigned) grid,kP2Threads,0,ctx->stream>>>(a);
  DX_LAUNCHED(ctx,"k_fa_pack2");
  return DX_OK;
}

int dxk_unpack2(dx_ctx *ctx, int kind, int upper, int width, const uint8_t *d_in, size_t n, const PkDecEntry *d_ent,
                int64_t count, const char *d_prefix, int plen, uint8_t *d_out, unsigned long long *d_ticket)
{ if (count == 0) return DX_OK;
  Unpack2Args a;
  a.kind = kind; a.upper = upper; a.width = width; a.in = d_in;
  a.in_end4 = d_in + ((n + 15) & ~(size_t) 15);
  a.ent = d_ent; a.count = count; a.prefix = d_prefix; a.plen = plen; a.out = d_out; a.ticket = d_ticket;
  int64_t grid = (count + kP2Warps - 1) / kP2Warps;
  if (grid > (int64_t) ctx->sm_count * 8) grid = (int64_t) ctx->sm_count * 8;
  DX_PROF_BEGIN(ctx); k_unpack2<<<(unsigned) grid,kP2Threads,0,ctx->stream>>>(a);
  DX_LAUNCHED(ctx,"k_unpack2");
  return DX_OK;
}

int dxk_pk_cand_prep(dx_ctx *ctx, const uint8_t *d_in, size_t n, size_t first, int fieldbytes, const int64_t *d_q,
                     int64_t count, int64_t *d_end, int32_t *d_ffrun, uint8_t *d_last)
{ if (count == 0) return DX_OK;
  DX_PROF_BEGIN(ctx);
  k_pk_cand_prep<<<(unsigned) ((count+255)/256),256,0,ctx->stream>>>(d_in,(int64_t) n,(int64_t) first,fieldbytes,d_q,count,
                                                                    d_end,d_ffrun,d_last);
  DX_LAUNCHED(ctx,"k_pk_cand_prep");
  return DX_OK;
}

int dxk_pk_layout(dx_ctx *ctx, int kind, const uint8_t *d_in, const int64_t *d_q, const int32_t *d_cand,
                  const int32_t *d_well, int64_t count, int fieldbytes, int plen, int width, uint32_t *d_len,
                  int64_t *d_opre, PkDecEntry *d_ent)
{ if (count > 0)
    { DX_PROF_BEGIN(ctx);
      k_pk_text_len<<<(unsigned) ((count+255)/256),256,0,ctx->stream>>>(kind,d_in,d_q,d_cand,d_well,count,plen,width,d_len);
      DX_LAUNCHED(ctx,"k_pk_text_len");
    }
  int rc = dxk_scan_u32(ctx,d_len,count,d_opre);
  if (rc != DX_OK) return rc;
  if (count > 0)
    { DX_PROF_BEGIN(ctx);
      k_pk_build_ent<<<(unsigned) ((count+255)/256),256,0,ctx->stream>>>(kind,d_in,d_q,d_cand,d_well,count,fieldbytes,width,
                                                                        d_opre,d_len,d_ent);
      DX_LAUNCHED(ctx,"k_pk_build_ent");
    }
  return DX_OK;
}

int dxk_compress_reads2(dx_ctx *ctx, int kind, const uint8_t *d_src, const int64_t *d_src_off,
                        const int32_t *d_len, int64_t nreads, uint8_t *d_dst, const int64_t *d_dst_off)
{ if (nreads == 0) return DX_OK;
  unsigned long long *d_ticket = (unsigned long long *) dx_arena_get(ctx,8);
  if (d_ticket == NULL) return DX_E_NOMEM;
  DX_CUDA(ctx,cudaMemsetAsync(d_ticket,0,8,ctx->stream));
  Reads2Args a;
  a.kind = kind; a.upper = 0; a.src = d_src; a.src_end4 = NULL; a.src_off = d_src_off; a.len = d_len; a.nreads = nreads;
  a.dst = d_dst; a.dst_off = d_dst_off; a.ticket = d_ticket;
  int64_t grid = (nreads + kP2Warps - 1) / kP2Warps;
  if (grid > (int64_t) ctx->sm_count * 8) grid = (int64_t) ctx->sm_count * 8;
  DX_PROF_BEGIN(ctx);
  if (kind == DX_FASTA) k_compress_reads2<DX_FASTA><<<(unsigned) grid,kP2Threads,0,ctx->stream>>>(a);
  else                  k_compress_reads2<DX_ARROW><<<(unsigned) grid,kP2Threads,0,ctx->stream>>>(a);
  DX_LAUNCHED(ctx,"k_compress_reads2");
  return DX_OK;
}

int dxk_uncompress_reads2(dx_ctx *ctx, int kind, int upper, const uint8_t *d_src,
                          const int64_t *d_src_off, const int32_t *d_len, int64_t nreads,
                          uint8_t *d_dst, const int64_t *d_dst_off)
{ if (nreads == 0) return DX_OK;
  unsigned long long *d_ticket = (unsigned long long *) dx_arena_get(ctx,8);
  if (d_ticket == NULL) return DX_E_NOMEM;
  DX_CUDA(ctx,cudaMemsetAsync(d_ticket,0,8,ctx->stream));
  Reads2Args a;
  a.kind = kind; a.upper = upper; a.src = d_src; a.src_end4 = NULL;
  a.src_off = d_src_off; a.len = d_len; a.nreads = nreads; a.dst = d_dst; a.dst_off = d_dst_off; a.ticket = d_ticket;
  int64_t grid = (nreads + kP2Warps - 1) / kP2Warps;
  if (grid > (int64_t) ctx->sm_count * 8) grid = (int64_t) ctx->sm_count * 8;
  DX_PROF_BEGIN(ctx); k_uncompress_reads2<<<(unsigned) grid,kP2Threads,0,ctx->stream>>>(a);
  DX_LAUNCHED(ctx,"k_uncompress_reads2");
  return DX_OK;
}
