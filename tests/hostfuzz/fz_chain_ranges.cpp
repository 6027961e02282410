// fz_chain_ranges.cpp -- the entry chain of a .dexqv image walked range after range, as
// dx_undexqv_range_* and the pipelined host decode walk it (CPU only, built with ASan + UBSan by
// tests/test_host_chain_ranges.py).
//
// An image is a header, then entries: delta bytes (0xff ... 0xff, d with d != 0xff; now and then a run
// of more than 4 KB), twelve field bytes, a payload of random bytes.  The image is cut at random
// offsets -- inside delta runs, fields, payloads, several cuts close together so that some ranges hold
// no entry start -- and every range [a, b) is walked by dx_chain_walk_general from the position and
// well the range before it ended at, seeing only what a range sees:
//   - candidates whose terminator lies in [a, b + 64) (the index of the range), true ones and false
//     ones (look-alikes in front of an entry, inside a payload, inside a delta run); some true ones
//     are missing (the filter missed them) or did not decode (cut short by their limit);
//   - 0xff runs counted no further back than a;
//   - the image bytes [a - 4096, buf_end) with buf_end a random tail behind b: a candidate that ends
//     behind buf_end did not decode; the slow path asks for more (as DX_E_CAP does) and the range is
//     walked again with the longer buffer.
// The slow path reads the delta bytes and the fields at the position it is given, and decodes "that
// entry alone": it must be a true entry -- reaching anything else is a failure.
// Checked: the ranges together give exactly the true entries and wells, end at n, every range stops at
// or behind its b and its last entry starts in front of it.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <map>
#include <vector>
#include <algorithm>
#include "dx_chain.h"

static uint64_t rng_state = 0x2545f4914f6cdd1dull;
static uint32_t rnd()
{ rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17;
  return (uint32_t) (rng_state >> 32);
}
static uint32_t rnd(uint32_t n) { return n ? rnd() % n : 0; }

struct Cand { int64_t q, end; bool truth; };

struct Slow                                   // what the slow path sees: the image up to buf_end
{ const std::vector<uint8_t> *img;
  const std::map<int64_t,int64_t> *ends;      // true entries: fields -> end
  int64_t buf_end, need;
  long calls;
};

static const int kShort = -2;                 // the stand-in for DX_E_CAP
static const int kWrong = -1;                 // the walk reached something that is no entry

static int slow(void *user, int64_t cur, int64_t *q, int64_t *end, int32_t *delta)
{ Slow *s = (Slow *) user;
  const std::vector<uint8_t> &img = *s->img;
  int64_t p = cur;
  int32_t add = 0;
  while (p < s->buf_end && img[(size_t) p] == 0xff) { add += 255; p++; }
  if (p >= s->buf_end) { s->need = p + 8421505; return kShort; }
  add += img[(size_t) p]; p++;
  const auto it = s->ends->find(p);
  if (it == s->ends->end()) return kWrong;
  if (p + 12 > s->buf_end || it->second > s->buf_end) { s->need = it->second; return kShort; }
  *q = p; *end = it->second; *delta = add;
  s->calls++;
  return 0;
}

int main(int argc, char **argv)
{ const int rounds = (argc > 1) ? atoi(argv[1]) : 20000;
  long nranges = 0, empty = 0, slow_entries = 0, retries = 0, long_runs = 0, straddles = 0;
  for (int round = 0; round < rounds; round++)
    { rng_state += 0x632be59bd9b4e019ull * (uint64_t) (round + 1);
      const int style = (int) rnd(4);
      std::vector<uint8_t> img;
      const int64_t first = 2 + (int64_t) rnd(5000);
      for (int64_t k = 0; k < first; k++) img.push_back((uint8_t) rnd(256));
      const int nent = 1 + (int) rnd(16);
      std::vector<Cand> cs;
      std::vector<int64_t> start, tq;
      std::vector<int32_t> twell;
      std::map<int64_t,int64_t> ends;
      int32_t well = (int32_t) rnd(1000);
      const int32_t well_in = well;
      for (int e = 0; e < nent; e++)
        { uint32_t delta = rnd(40);
          if (rnd(5) == 0) delta = 255 * (1 + rnd(4)) + rnd(255);
          if (style >= 2 && rnd(5) == 0) { delta = 255 * (4096 + rnd(3000)) + rnd(255); long_runs++; }   // > 4 KB of 0xff
          start.push_back((int64_t) img.size());
          for (uint32_t k = 0; k < delta / 255; k++) img.push_back(0xff);
          img.push_back((uint8_t) (delta % 255));
          well += (int32_t) delta;
          Cand c; c.q = (int64_t) img.size(); c.truth = true;
          for (int k = 0; k < 12; k++) img.push_back((uint8_t) rnd(256));
          const int plen = 4 * (int) (1 + rnd(style == 3 ? 3000 : 60));
          for (int k = 0; k < plen; k++) img.push_back((uint8_t) rnd(256));
          const int tail = (int) rnd(4);                   // a stream's last word may end in 0xff bytes
          for (int k = 0; k < tail; k++) img[img.size() - 1 - (size_t) k] = (rnd(2) == 0) ? 0xff : 0;
          c.end = (int64_t) img.size();
          cs.push_back(c); tq.push_back(c.q); twell.push_back(well);
          ends[c.q] = c.end;
        }
      const int64_t n = (int64_t) img.size();
      const int ntrue = (int) cs.size();
      for (int e = 0; e < ntrue; e++)                          // false candidates
        { for (int d = 4; d <= 8; d += 4)
            if (rnd(3) == 0 && cs[e].q - d > first + 1)
              { Cand f; f.q = cs[e].q - d; f.truth = false;
                f.end = (rnd(4) == 0) ? cs[e].end : f.q + 12 + (int64_t) rnd(200);
                cs.push_back(f);
              }
          if (rnd(3) == 0)
            { Cand f; f.q = cs[e].q + 1 + (int64_t) rnd((uint32_t) (cs[e].end - cs[e].q - 1)); f.truth = false;
              f.end = f.q + 12 + (int64_t) rnd(300);
              if (f.q + 12 <= n) cs.push_back(f);
            }
          if (rnd(3) == 0 && cs[e].q - 2 > first + 1)           // inside the delta run / the previous tail
            { Cand f; f.q = cs[e].q - 1 - (int64_t) rnd((uint32_t) std::min<int64_t>(cs[e].q - first - 2,6000)); f.truth = false;
              f.end = (rnd(2) == 0) ? cs[e].end : f.q + 12 + (int64_t) rnd(100);
              if (f.q > first + 1) cs.push_back(f);
            }
        }
      std::sort(cs.begin(),cs.end(),[](const Cand &x, const Cand &y) { return x.q < y.q || (x.q == y.q && x.truth > y.truth); });
      cs.erase(std::unique(cs.begin(),cs.end(),[](const Cand &x, const Cand &y) { return x.q == y.q; }),cs.end());
      // the filter's misses and the limit's cuts (fixed per image: every range sees the same)
      std::vector<bool> missed(cs.size()), cut(cs.size());
      for (size_t i = 0; i < cs.size(); i++)
        { missed[i] = cs[i].truth && style >= 1 && rnd(8) == 0;
          cut[i] = (style >= 1 && rnd(10) == 0);
        }

      // the cuts: random offsets, some inside delta runs, some close together
      std::vector<int64_t> cuts;
      const int ncut = 1 + (int) rnd(10);
      for (int k = 0; k < ncut; k++)
        { const uint32_t how = rnd(4);
          int64_t x;
          if (how == 0) { const int e = (int) rnd((uint32_t) ntrue); x = start[(size_t) e] + (int64_t) rnd((uint32_t) (tq[(size_t) e] - start[(size_t) e] + 14)); }
          else if (how == 1 && !cuts.empty()) x = cuts.back() + (int64_t) rnd(20);
          else x = (int64_t) rnd((uint32_t) n);
          cuts.push_back(std::min(std::max<int64_t>(x,0),n));
        }
      cuts.push_back(0); cuts.push_back(n);
      std::sort(cuts.begin(),cuts.end());

      int64_t cur = first;
      int32_t w = well_in;
      std::vector<int64_t> gotq;
      std::vector<int32_t> gotw;
      for (size_t r = 0; r + 1 < cuts.size(); r++)
        { const int64_t a = std::max(cuts[r],first), b = std::max(cuts[r+1],a);
          if (cur < a) { fprintf(stderr,"round %d: the chain stands at %lld, in front of the range [%lld, %lld)\n",round,
                                 (long long) cur,(long long) a,(long long) b); return 1; }
          int64_t buf_end = std::min(n,b + (int64_t) rnd(style == 3 ? 20000 : 600));
          for (int attempt = 0;; attempt++)
            { // what the range's index finds and the decode gives
              std::vector<int64_t> q, soff;
              std::vector<int32_t> ffrun, stat;
              std::vector<uint8_t> last;
              for (size_t i = 0; i < cs.size(); i++)
                { const int64_t t = cs[i].q - 1;
                  if (t < a || t >= b + 64 || cs[i].q + 12 > buf_end || missed[i]) continue;
                  q.push_back(cs[i].q);
                  last.push_back(img[(size_t) t]);
                  int32_t fr = 0;
                  for (int64_t k = t - 1; k >= a && img[(size_t) k] == 0xff; k--) fr++;
                  ffrun.push_back(fr);
                  const int64_t e = std::min(cs[i].end,n);
                  stat.push_back((cut[i] || e > buf_end) ? 1 : 0);
                  for (int k = 0; k < 6; k++) soff.push_back(e);
                }
              DxChainIn ci = { q.data(), ffrun.data(), last.data(), stat.data(), soff.data(), NULL, (int64_t) q.size(), a,
                               buf_end, cur, b };
              Slow s = { &img, &ends, buf_end, 0, 0 };
              std::vector<DxChainEntry> ent;
              int64_t stop = 0;
              const int rc = dx_chain_walk_general(ci,w,slow,&s,ent,&stop);
              if (rc == kShort)
                { if (s.need <= buf_end || attempt > 3)
                    { fprintf(stderr,"round %d: range [%lld, %lld) asks for %lld with a buffer to %lld\n",round,(long long) a,
                              (long long) b,(long long) s.need,(long long) buf_end); return 1; }
                  buf_end = std::min(n,s.need);
                  retries++;
                  continue;
                }
              if (rc != 0)
                { fprintf(stderr,"round %d: range [%lld, %lld) from %lld reached no entry (rc %d)\n",round,(long long) a,(long long) b,
                          (long long) cur,rc); return 1; }
              if (stop < b)
                { fprintf(stderr,"round %d: range [%lld, %lld) stopped at %lld\n",round,(long long) a,(long long) b,(long long) stop); return 1; }
              if (!ent.empty())
                { const int64_t last_start = (ent.size() > 1) ? ent[ent.size()-2].end : cur;
                  if (last_start >= b)
                    { fprintf(stderr,"round %d: range [%lld, %lld) took an entry that starts at %lld\n",round,(long long) a,
                              (long long) b,(long long) last_start); return 1; }
                  if (ent.back().q - 1 >= b) straddles++;
                }
              for (const DxChainEntry &e : ent)
                { gotq.push_back(e.q); gotw.push_back(e.well);
                  slow_entries += (e.cand < 0);
                }
              if (ent.empty()) empty++; else w = ent.back().well;
              cur = stop;
              nranges++;
              break;
            }
        }
      if (cur != n || gotq != tq || gotw != twell)
        { fprintf(stderr,"round %d: the ranges found %zu entries and ended at %lld; the image has %d and ends at %lld\n",round,
                  gotq.size(),(long long) cur,ntrue,(long long) n);
          for (size_t k = 0; k < std::min(gotq.size(),tq.size()); k++)
            if (gotq[k] != tq[k] || gotw[k] != twell[k])
              { fprintf(stderr,"  entry %zu: fields %lld well %d, want %lld well %d\n",k,(long long) gotq[k],gotw[k],
                        (long long) tq[k],twell[k]); break; }
          return 1;
        }
    }
  printf("ok %d images: %ld ranges, %ld without an entry, %ld entries by the slow path, %ld longer buffers, "
         "%ld delta runs over 4 KB, %ld entries whose fields lie behind their range\n",
         rounds,nranges,empty,slow_entries,retries,long_runs,straddles);
  return 0;
}
