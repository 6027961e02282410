// dx_pack.cu -- the 2-bit codec on the device: .fasta <-> .dexta and .arrow <-> .dexar.
//
// Replaces Number_Read / Number_Arrow + Compress_Read (reference DB.c:393-441, 319-338) for every
// entry of a file at once, and Uncompress_Read + Lower_/Upper_Read / Letter_Arrow
// (DB.c:342-389) with the line wrapping of undexta.c:263-270.
//
//   k_fa_measure  one warp per entry: header fields, first sequence character, exact symbol
//                 count (region bytes minus newlines), line width, regularity of the line layout
//   k_fa_offsets  exclusive scan of encoded entry sizes (well-delta bytes + fields + payload)
//   k_fa_pack     one warp per entry: 16 symbols -> one 32-bit word per lane, staged in shared
//                 memory and flushed at the payload's byte alignment; irregular entries (ragged
//                 line widths) take a sequential per-entry path in the same kernel
//   k_unpack      one warp per entry: header text, then 16 output characters per lane per step

#include "dx_internal.h"
#include "dx_common.cuh"

namespace {

constexpr int kPkWarps   = 8;
constexpr int kPkThreads = kPkWarps * 32;
constexpr int kLineLimit = 99998;             // dexta.c:21,168: MAX_BUFFER-2 characters per line

__device__ __forceinline__ uint32_t code_of(int kind, uint32_t c)
{ if (kind == DX_FASTA)                       // DB.c:394-411
    { c |= 0x20u;
      return (c == 'c') ? 1u : (c == 'g') ? 2u : (c == 't') ? 3u : 0u;
    }
  // DB.c:419-436: '1','2','3' -> 0,1,2 ; 'G' -> 2 ; everything else (incl. '4') -> 3
  return (c == '1') ? 0u : (c == '2') ? 1u : (c == '3' || c == 'G') ? 2u : 3u;
}

__device__ __forceinline__ bool digits(const uint8_t *t, int64_t &p, int64_t end, int32_t &val)
{ int64_t s = p;
  uint32_t v = 0;
  while (p < end && t[p] >= '0' && t[p] <= '9' && p - s < 9)
    v = v*10 + (t[p++] - '0');
  if (p == s || (p < end && t[p] >= '0' && t[p] <= '9')) return false;
  val = (int32_t) v;
  return true;
}

// canonical two-decimal SNR "d+.dd" -> the uint16 the reference stores (dexar.c:152-163)
__device__ __forceinline__ bool snr_field(const uint8_t *t, int64_t &p, int64_t end, uint32_t &cnr)
{ int32_t ip = 0;
  if (!digits(t,p,end,ip) || ip > 99999) return false;
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
__device__ bool parse_header(int kind, const uint8_t *t, int64_t p, int64_t end,
                             int32_t &well, int32_t &beg, int32_t &en, int32_t aux[2])
{ p += 1;
  while (p < end && t[p] != '/') p++;
  if (p >= end) return false;
  p++;
  if (!digits(t,p,end,well) || p >= end || t[p] != '/') return false;
  p++;
  if (!digits(t,p,end,beg) || p >= end || t[p] != '_') return false;
  p++;
  if (!digits(t,p,end,en)) return false;
  if (kind == DX_FASTA)
    { aux[0] = aux[1] = 0;
      if (p == end) return true;                                     // no RQ field: qv = 0
      if (p + 6 > end || t[p] != ' ' || t[p+1] != 'R' || t[p+2] != 'Q' || t[p+3] != '=' ||
          t[p+4] != '0' || t[p+5] != '.') return false;
      p += 6;
      return digits(t,p,end,aux[0]);
    }
  if (p + 4 > end || t[p] != ' ' || t[p+1] != 'S' || t[p+2] != 'N' || t[p+3] != '=') return false;
  p += 4;
  uint32_t c[4];
  for (int k = 0; k < 4; k++)
    { if (!snr_field(t,p,end,c[k])) return false;
      if (k < 3) { if (p >= end || t[p] != ',') return false; p++; }
    }
  aux[0] = (int32_t) (c[0] | (c[1] << 16));
  aux[1] = (int32_t) (c[2] | (c[3] << 16));
  return true;
}

// ---- measure ------------------------------------------------------------------------------------

__global__ void __launch_bounds__(kPkThreads)
k_fa_measure(int kind, const uint8_t *text, int64_t n, const int64_t *hdr, FaEntries ent)
{ const int lane = threadIdx.x & 31;
  const int64_t nwarp = ((int64_t) gridDim.x * blockDim.x) >> 5;
  for (int64_t e = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5; e < ent.n; e += nwarp)
    { const int64_t h0 = hdr[e];
      const int64_t stop = (e+1 < ent.n) ? hdr[e+1] : n;
      // end of the header line
      int64_t h1 = -1;
      for (int64_t b = h0; b < stop && h1 < 0; b += 32)
        { bool nl = (b + lane < stop) && text[b + lane] == '\n';
          uint32_t m = __ballot_sync(DX_FULL,nl);
          if (m) h1 = b + __ffs(m) - 1;
        }
      int32_t flag = 0;
      if (h1 < 0) { h1 = stop - 1; flag |= 4; }                     // unterminated header line
      if (h1 - h0 > kLineLimit) flag |= 4;
      const int64_t seq = h1 + 1, region = stop - seq;

      // newlines of the sequence region: count, first, and whether they sit on a W+1 lattice
      const uint8_t *r0 = text + seq;
      const int skew = (int) (reinterpret_cast<uintptr_t>(r0) & 15);
      const uint8_t *base = r0 - skew;
      const int64_t nchunk = (skew + region + 15) >> 4;
      int64_t first_nl = -1;
      // pass A: first newline (defines the width)
      for (int64_t c0 = 0; c0 < nchunk && first_nl < 0; c0 += 32)
        { const int64_t c = c0 + lane;
          uint32_t m = 0;
          if (c < nchunk)
            { const int64_t p0 = c*16 - skew;
              const int lo = (int) max((int64_t) 0,-p0), hi = (int) min((int64_t) 16,region - p0);
              m = dx_eq_mask16(dx_ldg16(base + c*16),'\n') & dx_range16(lo,hi);
            }
          const uint32_t any = __ballot_sync(DX_FULL,m != 0);
          if (any)
            { const int src = __ffs(any) - 1;
              const uint32_t mm = __shfl_sync(DX_FULL,m,src);
              first_nl = (c0 + src)*16 - skew + (__ffs(mm) - 1);
            }
        }
      const int64_t W = (first_nl < 0) ? region : first_nl;        // first line length
      uint32_t nl_count = 0, off_lattice = 0;
      int64_t last_nl = -1;                                         // region offset of the last newline so far
      bool toolong = false;                                         // a line of more than kLineLimit characters
      for (int64_t c0 = 0; c0 < nchunk; c0 += 32)
        { const int64_t c = c0 + lane;
          uint32_t m0 = 0;
          if (c < nchunk)
            { const int64_t p0 = c*16 - skew;
              const int lo = (int) max((int64_t) 0,-p0), hi = (int) min((int64_t) 16,region - p0);
              m0 = dx_eq_mask16(dx_ldg16(base + c*16),'\n') & dx_range16(lo,hi);
            }
          // dexta.c:168-172: no line may have more than MAX_BUFFER-2 characters.  Inside a round of
          // 512 bytes no gap can; what can is the gap back to the last newline of an earlier round.
          { const uint32_t any = __ballot_sync(DX_FULL,m0 != 0);
            if (any)
              { const int f = __ffs(any) - 1, l = 31 - __clz(any);
                const int64_t first = (c0 + f)*16 - skew + (__ffs(__shfl_sync(DX_FULL,m0,f)) - 1);
                if (first - last_nl - 1 > kLineLimit) toolong = true;
                last_nl = (c0 + l)*16 - skew + (31 - __clz(__shfl_sync(DX_FULL,m0,l)));
              }
          }
          if (c < nchunk)
            { const int64_t p0 = c*16 - skew;
              uint32_t m = m0;
              nl_count += __popc(m);
              while (m)
                { const int i = __ffs(m) - 1; m &= m - 1;
                  const int64_t q = p0 + i;                          // region offset of this '\n'
                  if ((q + 1) % (W + 1) != 0 && q != region - 1) off_lattice++;
                }
            }
        }
      nl_count    = dx_warp_sum(nl_count);
      off_lattice = dx_warp_sum(off_lattice);
      if (region > 0 && text[stop-1] != '\n') flag |= 4;            // last line unterminated
      if (off_lattice) flag |= 2;
      if (W > kLineLimit || toolong || region - last_nl - 1 > kLineLimit) flag |= 4;
      const int64_t rlen = region - nl_count;
      if (rlen >= (int64_t) 1 << 30) flag |= 4;
      // regular = every line but the last has exactly W symbols and the last has 1..W
      if (rlen > 0 && (W == 0 || !((int64_t) (nl_count-1)*W < rlen && rlen <= (int64_t) nl_count*W)))
        flag |= 2;

      if (lane == 0)
        { int32_t well = 0, beg = 0, en = 0, aux[2] = { 0, 0 };
          if (text[h0] != '>' || !parse_header(kind,text,h0,h1,well,beg,en,aux)) flag |= 1;
          ent.hdr[e] = h0; ent.seq[e] = seq; ent.region[e] = region;
          ent.rlen[e] = (int32_t) rlen; ent.width[e] = (int32_t) min(W,(int64_t) 0x7fffffff);
          ent.well[e] = well; ent.beg[e] = beg; ent.end[e] = en;
          ent.aux[2*e] = aux[0]; ent.aux[2*e+1] = aux[1];
          ent.flag[e] = flag;
        }
    }
}

// ---- offsets --------------------------------------------------------------------------------------

// encoded bytes of every entry: well-delta bytes + fields + payload (dexta.c:187-204); the offsets
// are their exclusive scan (dxk_scan_u32)
__global__ void k_fa_bytes(int kind, FaEntries ent, int32_t lwell_in)
{ const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ent.n) return;
  const uint32_t fields = (kind == DX_FASTA) ? 12u : 16u;
  const int32_t lw = (i == 0) ? lwell_in : ent.well[i-1];
  const int32_t d  = ent.well[i] - lw;
  const uint32_t wb = 1u + (d >= 255 ? (uint32_t) d / 255u : 0u);
  ent.bytes[i] = wb + fields + (((uint32_t) ent.rlen[i] + 3u) >> 2);
}

// ---- pack -------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(kPkThreads)
k_fa_pack(int kind, const uint8_t *text, FaEntries ent, int32_t lwell_in, uint8_t *out)
{ __shared__ uint32_t stage_all[kPkWarps][36];
  const int lane = threadIdx.x & 31;
  uint32_t *stage = stage_all[threadIdx.x >> 5];
  const int64_t nwarp = ((int64_t) gridDim.x * blockDim.x) >> 5;
  const uint32_t fields = (kind == DX_FASTA) ? 12u : 16u;

  for (int64_t e = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5; e < ent.n; e += nwarp)
    { const int32_t rlen = ent.rlen[e];
      const int64_t W    = ent.width[e];
      const uint8_t *seq = text + ent.seq[e];
      uint8_t *dst = out + ent.off[e];

      // entry header: well-delta bytes, beg, end, qv | 4 x uint16 SNR (dexta.c:187-198)
      if (lane == 0)
        { int32_t lwell = (e == 0) ? lwell_in : ent.well[e-1];
          const int32_t well = ent.well[e];
          uint8_t *h = dst;
          while (well - lwell >= 255) { *h++ = 0xff; lwell += 255; }
          *h++ = (uint8_t) (well - lwell);
          const uint32_t f[4] = { (uint32_t) ent.beg[e], (uint32_t) ent.end[e],
                                  (uint32_t) ent.aux[2*e], (uint32_t) ent.aux[2*e+1] };
          for (uint32_t k = 0; k < fields; k++)
            *h++ = (uint8_t) (f[k >> 2] >> (8*(k & 3)));
        }
      uint8_t *pay = dst + (ent.bytes[e] - (((uint32_t) rlen + 3u) >> 2));

      if (ent.flag[e] & 2)
        { // ragged line layout: one lane walks the region (rare; dexta.c:161-183 semantics)
          if (lane == 0)
            { const int64_t region = ent.region[e];
              uint32_t acc = 0, cnt = 0;
              for (int64_t q = 0; q < region; q++)
                { const uint32_t c = seq[q];
                  if (c == '\n') continue;
                  acc = (acc << 2) | code_of(kind,c);
                  if (++cnt == 4) { *pay++ = (uint8_t) acc; acc = 0; cnt = 0; }
                }
              if (cnt) *pay = (uint8_t) (acc << (2*(4-cnt)));
            }
          __syncwarp();
          continue;
        }

      // regular layout: symbol b sits at region offset b + b/W
      const int64_t nword = ((int64_t) rlen + 15) >> 4;               // 16 symbols per word
      for (int64_t w0 = 0; w0 < nword; w0 += 32)
        { const int64_t w = w0 + lane;
          uint32_t val = 0;
          if (w < nword)
            { const int32_t b = (int32_t) (w*16);                       // rlen < 2^30
              const int32_t line = (W > 0) ? b / (int32_t) W : 0;
              int32_t col  = b - line*(int32_t) W;
              const uint8_t *p = seq + b + line;
              const int cnt = min(16,rlen - b);
              for (int k = 0; k < cnt; k++)
                { val |= code_of(kind,*p) << (30 - 2*k);
                  p++;
                  if (++col == (int32_t) W) { col = 0; p++; }         // step over the '\n'
                }
              val = __byte_perm(val,0,0x0123);                        // first symbol -> first byte
            }
          stage[lane] = val;
          __syncwarp();
          const int64_t nb = min((int64_t) 128,(((int64_t) rlen + 3) >> 2) - w0*4);
          dx_warp_copy_out(pay + w0*4,stage,(uint32_t) nb,lane);
          __syncwarp();
        }
    }
}

// ---- walk of a 2-bit image ----------------------------------------------------------------------------

__global__ void k_pk_walk(int fieldbytes, const uint8_t *in, int64_t n, const int64_t *q,
                          int64_t count, int64_t *end)
{ const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const uint8_t *p = in + q[i];
  const uint32_t beg = (uint32_t) p[0] | ((uint32_t) p[1] << 8) | ((uint32_t) p[2] << 16) | ((uint32_t) p[3] << 24);
  const uint32_t en  = (uint32_t) p[4] | ((uint32_t) p[5] << 8) | ((uint32_t) p[6] << 16) | ((uint32_t) p[7] << 24);
  const int64_t rlen = (int64_t) (int32_t) (en - beg);
  int64_t stop = q[i] + fieldbytes + ((rlen + 3) >> 2);
  end[i] = (rlen < 0 || stop > n) ? -1 : stop;
}

// ---- unpack -------------------------------------------------------------------------------------------

__device__ int fmt_int(uint8_t *p, int32_t v)
{ char tmp[12];
  int  k = 0, len = 0;
  uint32_t u = (v < 0) ? (uint32_t) (-(int64_t) v) : (uint32_t) v;
  if (v < 0) p[len++] = '-';
  do { tmp[k++] = (char) ('0' + u % 10); u /= 10; } while (u);
  while (k) p[len++] = (uint8_t) tmp[--k];
  return len;
}

__global__ void __launch_bounds__(kPkThreads)
k_unpack(int kind, int upper, int width, const uint8_t *in, const PkDecEntry *ent, int64_t count,
         const char *prefix, int plen, uint8_t *out)
{ __shared__ uint32_t stage_all[kPkWarps][132];
  const int lane = threadIdx.x & 31;
  uint32_t *stage = stage_all[threadIdx.x >> 5];
  const int64_t nwarp = ((int64_t) gridDim.x * blockDim.x) >> 5;
  const uint32_t alpha = (kind == DX_ARROW) ? 0x34333231u          // "1234"
                        : upper ? 0x54474341u : 0x74676361u;       // "ACGT" / "acgt"
  const int64_t W = width;

  for (int64_t e = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5; e < count; e += nwarp)
    { const PkDecEntry en = ent[e];
      const int64_t rlen = (int64_t) en.end - en.beg;
      if (lane == 0)
        { // "%s/%d/%d_%d RQ=0.%d\n" (undexta.c:242) or " SN=%.2f,%.2f,%.2f,%.2f\n" (undexar.c:202)
          uint8_t *h = out + en.out_off;
          int hl = 0;
          for (int k = 0; k < plen; k++) h[hl++] = (uint8_t) prefix[k];
          h[hl++] = '/'; hl += fmt_int(h+hl,en.well);
          h[hl++] = '/'; hl += fmt_int(h+hl,en.beg);
          h[hl++] = '_'; hl += fmt_int(h+hl,en.end);
          if (kind == DX_FASTA)
            { const char *rq = " RQ=0.";
              for (int k = 0; k < 6; k++) h[hl++] = (uint8_t) rq[k];
              hl += fmt_int(h+hl,en.aux[0]);
            }
          else
            { const char *sn = " SN=";
              for (int k = 0; k < 4; k++) h[hl++] = (uint8_t) sn[k];
              for (int k = 0; k < 4; k++)
                { const uint32_t c = ((uint32_t) en.aux[k >> 1] >> (16*(k & 1))) & 0xffffu;
                  hl += fmt_int(h+hl,(int32_t) (c / 100u));
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
      const int64_t nlines = (rlen + W - 1) / W;
      const int64_t tlen = rlen + nlines;
      const uint8_t *pay = in + en.bin_off;
      uint8_t *dst = out + en.text_off;
      for (int64_t t0 = 0; t0 < tlen; t0 += 512)
        { // lane produces text bytes [t0 + 16*lane, +16)
          const int64_t tb = t0 + 16*lane;
          uint32_t wv[4] = { 0, 0, 0, 0 };
          if (tb < tlen)
            { int64_t line = tb / (W + 1);
              int64_t col  = tb - line*(W + 1);                      // col == W  <=> newline slot
              int64_t b    = line*W + col;                           // symbol index (if col < W)
              const int cnt = (int) min((int64_t) 16,tlen - tb);
              for (int k = 0; k < cnt; k++)
                { uint32_t ch;
                  if (col == W || b >= rlen)
                    { ch = '\n'; col = 0; }
                  else
                    { const uint32_t byte = pay[b >> 2];
                      ch = (alpha >> (8*((byte >> (6 - 2*(b & 3))) & 3u))) & 0xffu;
                      b++; col++;
                    }
                  wv[k >> 2] |= ch << (8*(k & 3));
                }
            }
          stage[4*lane] = wv[0]; stage[4*lane+1] = wv[1]; stage[4*lane+2] = wv[2]; stage[4*lane+3] = wv[3];
          __syncwarp();
          const int64_t nb = min((int64_t) 512,tlen - t0);
          dx_warp_copy_out(dst + t0,stage,(uint32_t) nb,lane);
          __syncwarp();
        }
    }
}

// ---- batched in-memory reads (no line structure) -------------------------------------------------------

__global__ void __launch_bounds__(kPkThreads)
k_compress_reads(int kind, const uint8_t *src, const int64_t *src_off, const int32_t *len,
                 int64_t nreads, uint8_t *dst, const int64_t *dst_off)
{ __shared__ uint32_t stage_all[kPkWarps][36];
  const int lane = threadIdx.x & 31;
  uint32_t *stage = stage_all[threadIdx.x >> 5];
  const int64_t nwarp = ((int64_t) gridDim.x * blockDim.x) >> 5;
  for (int64_t r = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < nreads; r += nwarp)
    { const int32_t rlen = len[r];
      const uint8_t *s = src + src_off[r];
      uint8_t *pay = dst + dst_off[r];
      const int32_t nword = (rlen + 15) >> 4;
      for (int32_t w0 = 0; w0 < nword; w0 += 32)
        { const int32_t w = w0 + lane;
          uint32_t val = 0;
          if (w < nword)
            { const int cnt = min(16,rlen - w*16);
              for (int k = 0; k < cnt; k++)
                val |= code_of(kind,s[w*16 + k]) << (30 - 2*k);
              val = __byte_perm(val,0,0x0123);
            }
          stage[lane] = val;
          __syncwarp();
          const int32_t nb = min(128,((rlen + 3) >> 2) - w0*4);
          dx_warp_copy_out(pay + (int64_t) w0*4,stage,(uint32_t) nb,lane);
          __syncwarp();
        }
    }
}

__global__ void __launch_bounds__(kPkThreads)
k_uncompress_reads(int kind, int upper, const uint8_t *src, const int64_t *src_off,
                   const int32_t *len, int64_t nreads, uint8_t *dst, const int64_t *dst_off)
{ __shared__ uint32_t stage_all[kPkWarps][132];
  const int lane = threadIdx.x & 31;
  uint32_t *stage = stage_all[threadIdx.x >> 5];
  const int64_t nwarp = ((int64_t) gridDim.x * blockDim.x) >> 5;
  const uint32_t alpha = (kind == DX_ARROW) ? 0x34333231u : upper ? 0x54474341u : 0x74676361u;
  for (int64_t r = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < nreads; r += nwarp)
    { const int32_t rlen = len[r];
      const uint8_t *pay = src + src_off[r];
      uint8_t *out = dst + dst_off[r];
      for (int32_t t0 = 0; t0 < rlen; t0 += 512)
        { const int32_t tb = t0 + 16*lane;
          uint32_t wv[4] = { 0, 0, 0, 0 };
          if (tb < rlen)
            { const int cnt = min(16,rlen - tb);
              uint32_t pk = 0;
              for (int k = 0; k < (cnt + 3) >> 2; k++)
                pk |= (uint32_t) pay[(tb >> 2) + k] << (8*k);
              for (int k = 0; k < cnt; k++)
                { const uint32_t byte = (pk >> (8*(k >> 2))) & 0xffu;
                  const uint32_t ch = (alpha >> (8*((byte >> (6 - 2*(k & 3))) & 3u))) & 0xffu;
                  wv[k >> 2] |= ch << (8*(k & 3));
                }
            }
          stage[4*lane] = wv[0]; stage[4*lane+1] = wv[1]; stage[4*lane+2] = wv[2]; stage[4*lane+3] = wv[3];
          __syncwarp();
          dx_warp_copy_out(out + t0,stage,(uint32_t) min(512,rlen - t0),lane);
          __syncwarp();
        }
    }
}

}  // namespace

int dxk_compress_reads(dx_ctx *ctx, int kind, const uint8_t *d_src, const int64_t *d_src_off,
                       const int32_t *d_len, int64_t nreads, uint8_t *d_dst, const int64_t *d_dst_off)
{ if (nreads == 0) return DX_OK;
  DX_PROF_BEGIN(ctx); k_compress_reads<<<ctx->sm_count*8,kPkThreads,0,ctx->stream>>>(kind,d_src,d_src_off,d_len,nreads,d_dst,d_dst_off);
  DX_LAUNCHED(ctx,"k_compress_reads");
  return DX_OK;
}

int dxk_uncompress_reads(dx_ctx *ctx, int kind, int upper, const uint8_t *d_src,
                         const int64_t *d_src_off, const int32_t *d_len, int64_t nreads,
                         uint8_t *d_dst, const int64_t *d_dst_off)
{ if (nreads == 0) return DX_OK;
  DX_PROF_BEGIN(ctx); k_uncompress_reads<<<ctx->sm_count*8,kPkThreads,0,ctx->stream>>>(kind,upper,d_src,d_src_off,d_len,nreads,d_dst,d_dst_off);
  DX_LAUNCHED(ctx,"k_uncompress_reads");
  return DX_OK;
}

int dxk_fa_measure(dx_ctx *ctx, int kind, const uint8_t *d_text, size_t n, const int64_t *d_hdr,
                   FaEntries ent)
{ if (ent.n == 0) return DX_OK;
  const int grid = ctx->sm_count * 8;
  DX_PROF_BEGIN(ctx); k_fa_measure<<<grid,kPkThreads,0,ctx->stream>>>(kind,d_text,(int64_t) n,d_hdr,ent);
  DX_LAUNCHED(ctx,"k_fa_measure");
  return DX_OK;
}

int dxk_fa_offsets(dx_ctx *ctx, int kind, FaEntries ent, int32_t lwell_in, int64_t *h_total)
{ *h_total = 0;
  if (ent.n == 0) return DX_OK;
  DX_PROF_BEGIN(ctx); k_fa_bytes<<<(unsigned) ((ent.n + 255)/256),256,0,ctx->stream>>>(kind,ent,lwell_in);
  DX_LAUNCHED(ctx,"k_fa_bytes");
  int rc = dxk_scan_u32(ctx,ent.bytes,ent.n,ent.off);
  if (rc != DX_OK) return rc;
  DX_CUDA(ctx,cudaMemcpyAsync(h_total,ent.off+ent.n,8,cudaMemcpyDeviceToHost,ctx->stream));
  DX_CUDA(ctx,cudaStreamSynchronize(ctx->stream));
  return DX_OK;
}

int dxk_fa_pack(dx_ctx *ctx, int kind, const uint8_t *d_text, size_t n, FaEntries ent,
                int32_t lwell_in, uint8_t *d_out)
{ (void) n;
  if (ent.n == 0) return DX_OK;
  const int grid = ctx->sm_count * 8;
  DX_PROF_BEGIN(ctx); k_fa_pack<<<grid,kPkThreads,0,ctx->stream>>>(kind,d_text,ent,lwell_in,d_out);
  DX_LAUNCHED(ctx,"k_fa_pack");
  return DX_OK;
}

int dxk_pk_walk(dx_ctx *ctx, int fieldbytes, const uint8_t *d_in, size_t n, const int64_t *d_q,
                int64_t count, int64_t *d_end)
{ if (count == 0) return DX_OK;
  DX_PROF_BEGIN(ctx); k_pk_walk<<<(unsigned) ((count+255)/256),256,0,ctx->stream>>>(fieldbytes,d_in,(int64_t) n,d_q,count,d_end);
  DX_LAUNCHED(ctx,"k_pk_walk");
  return DX_OK;
}

int dxk_unpack(dx_ctx *ctx, int kind, int upper, int width, const uint8_t *d_in,
               const PkDecEntry *d_ent, int64_t count, const char *d_prefix, int plen,
               uint8_t *d_out)
{ if (count == 0) return DX_OK;
  const int grid = ctx->sm_count * 8;
  DX_PROF_BEGIN(ctx); k_unpack<<<grid,kPkThreads,0,ctx->stream>>>(kind,upper,width,d_in,d_ent,count,d_prefix,plen,d_out);
  DX_LAUNCHED(ctx,"k_unpack");
  return DX_OK;
}
