// dx_chain.h -- which candidates of a .dexqv image are its entries.
//
// undexqv.c:119-208 reads one entry after the other: the well-delta bytes (0xff ... 0xff, d with
// d != 0xff), the fields, the five streams -- and whatever follows the last stream is the next
// entry.  The image stores no entry lengths, so a whole-file decoder has to find the entry starts.
// Every offset whose next 12 bytes look like beg/end/qv is a CANDIDATE (k_pred_slots<QVCAND>); all
// candidates are decoded at once, which gives every one of them an end; this file decides, from the
// candidates' positions, ends and the bytes in front of their fields, which of them form the chain
// the reference would walk.  Two forms of the same decision:
//
//   dx_chain_walk       the walk itself, on the host, O(candidates): candidate i is the next entry
//                       iff the bytes between the end of the previous entry and its fields are
//                       exactly its delta bytes;
//   dx_chain_check_one  the same decision as a predicate per candidate, for the case in which the
//                       text was laid out in advance for a chosen subset (keep[]) with every delta
//                       but the first below 255: there IS a kept candidate and ALL of them pass  <=>
//                       the walk accepts exactly the kept candidates with no 0xff delta byte except
//                       in front of the first (tests/hostfuzz/fz_chain.cpp drives both on random
//                       images; it found the "there is one" half);
//   dx_chain_walk_general  the walk over one byte range of an image, which has no whole image to fall
//                       back to: where the candidates break the chain, the entry is read by a slow path
//                       (tests/hostfuzz/fz_chain_ranges.cpp walks random images range after range).
//
// Plain C++ (no CUDA types) so that the host, the kernel (dx_qv_plan.cu) and the fuzz harness share it.

#ifndef DX_CHAIN_H
#define DX_CHAIN_H

#include <stdint.h>
#include <vector>

#if defined(__CUDACC__)
#define DX_CHAIN_HD __host__ __device__ __forceinline__
#else
#define DX_CHAIN_HD static inline
#endif

struct DxChainIn
{ const int64_t *q;        // [N] position of the fields (the terminator byte is at q-1), ascending
  const int32_t *ffrun;    // [N] 0xff bytes directly in front of the terminator (not reaching below `first`)
  const uint8_t *last;     // [N] the terminator byte
  const int32_t *stat;     // [N] != 0: the candidate did not decode
  const int64_t *soff;     // [N][6] stream offsets of the decode; [5] = first byte behind the entry
  const uint8_t *keep;     // [N] part of the layout assumed in advance (NULL: nothing was assumed)
  int64_t N, first, n;     // candidates, first byte behind the coding header, bytes every entry ends within
  int64_t start = first,   // the walk's first entry and its bound (entries start below it); left out: the
          stop = n;        // whole image
};

// One step of the reference's loop for every entry that starts in [start, stop).  cand[m] / well[m]
// (m < *M): the candidate that is entry m and its well number.  *as_assumed: the entries are exactly
// the kept candidates and no entry but the first has 0xff delta bytes.  *cur_out (if asked for): where
// the next entry starts (windows that carry it and the last well walk the chain of one whole walk).
// Returns false when the chain breaks (an entry the candidates miss, a candidate that did not decode):
// the caller takes the general path.
static inline bool dx_chain_walk(const DxChainIn &c, int32_t well_in, int32_t *cand, int32_t *well_out,
                                 int64_t *M_out, bool *as_assumed, int64_t *cur_out = NULL)
{ int64_t M = 0, kept = 0;
  bool same = true;
  if (c.keep != NULL)
    for (int64_t i = 0; i < c.N; i++) kept += (c.keep[i] != 0);
  int64_t cur = c.start, i = 0;
  int32_t well = well_in;
  while (cur < c.stop)
    { while (i < c.N && c.q[i] - 1 < cur) i++;
      // a candidate whose terminator byte is 0xff is no terminator: part of a longer delta
      while (i < c.N && c.last[i] == 0xff && c.q[i] - 1 - cur <= c.ffrun[i]) i++;
      if (i >= c.N || c.stat[i] != 0) return false;
      const int64_t gap = c.q[i] - 1 - cur;
      if (gap > c.ffrun[i] || c.last[i] == 0xff) return false;
      const int64_t end = c.soff[6*i + 5];
      if (end > c.n || end <= cur) return false;
      if (c.keep == NULL || !c.keep[i] || (gap != 0 && !(M == 0 && gap == c.ffrun[i]))) same = false;
      well += 255 * (int32_t) gap + c.last[i];
      cand[M] = (int32_t) i; well_out[M] = well; M++;
      cur = end;
      i++;
    }
  if (M != kept) same = false;
  *M_out = M;
  *as_assumed = same;
  if (cur_out != NULL) *cur_out = cur;
  return true;
}

// The walk without a way out, for a caller that has no whole image to fall back to (one byte range of
// an image, dx_undexqv_range_*): wherever dx_chain_walk would return false, the entry at cur is taken
// from `slow`, which reads its delta bytes and fields at cur and decodes that one entry by itself (the
// reference's loop for a single entry): *q its fields, *end the first byte behind it (> cur), *delta
// its well delta.  A candidate the filter missed, one whose speculative decode was cut short, a 0xff
// run whose terminator lies beyond the candidates: none of them stops the walk.  Entry m is ent[m]
// (cand -1: found by `slow`).  Returns 0, or the first non-zero status of `slow`.
struct DxChainEntry { int64_t q, end; int32_t cand, well; };
typedef int (*DxChainSlow)(void *user, int64_t cur, int64_t *q, int64_t *end, int32_t *delta);

static inline int dx_chain_walk_general(const DxChainIn &c, int32_t well_in, DxChainSlow slow, void *user,
                                        std::vector<DxChainEntry> &ent, int64_t *cur_out)
{ int64_t cur = c.start, i = 0;
  int32_t well = well_in;
  ent.clear();
  while (cur < c.stop)
    { while (i < c.N && c.q[i] - 1 < cur) i++;
      while (i < c.N && c.last[i] == 0xff && c.q[i] - 1 - cur <= c.ffrun[i]) i++;
      DxChainEntry e;
      const int64_t gap = (i < c.N) ? c.q[i] - 1 - cur : 0;
      if (i < c.N && c.stat[i] == 0 && gap <= c.ffrun[i] && c.last[i] != 0xff &&
          c.soff[6*i + 5] <= c.n && c.soff[6*i + 5] > cur)
        { e.q = c.q[i]; e.end = c.soff[6*i + 5]; e.cand = (int32_t) i;
          well += 255 * (int32_t) gap + c.last[i];
          i++;
        }
      else
        { int32_t delta = 0;
          const int rc = slow(user,cur,&e.q,&e.end,&delta);
          if (rc != 0) return rc;
          e.cand = -1;
          well += delta;
        }
      e.well = well;
      ent.push_back(e);
      cur = e.end;
    }
  *cur_out = cur;
  return 0;
}

// Kept candidate i confirms the assumed layout: it decoded, its terminator is one, it ends exactly
// where the terminator of the next kept candidate stands (at the image's end if it is the last),
// and if it is the first kept one its terminator is the first byte behind the header or has only
// 0xff bytes between the header and itself.  rlen_d[i] < 0: left out of the decode (cannot fit).
DX_CHAIN_HD bool dx_chain_check_one(const DxChainIn &c, const int32_t *rlen_d, int64_t i)
{ bool ok = (rlen_d[i] >= 0 && c.stat[i] == 0 && c.last[i] != 0xff);
  int64_t j = i + 1;                                    // next kept candidate
  while (j < c.N && !c.keep[j]) j++;
  const int64_t end = c.soff[6*i + 5];
  ok = ok && (end == ((j < c.N) ? c.q[j] - 1 : c.n));
  int64_t k = i - 1;                                    // the first kept one? (only dropped ones in front:
  while (k >= 0 && !c.keep[k]) k--;                     //  the walk ends at once everywhere else)
  if (k < 0) ok = ok && (c.q[i] - 1 - c.first == 0 || c.q[i] - 1 - c.first == (int64_t) c.ffrun[i]);
  return ok;
}

#endif
