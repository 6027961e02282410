// fz_chain.cpp -- the two forms of the entry-chain decision of dx_chain.h on random .dexqv-like
// images (CPU only, built with ASan + UBSan by tests/test_host_sanitizers.py).
//
// An image is a header, then entries: delta bytes (0xff ... 0xff, d with d != 0xff), twelve field
// bytes, a payload of random bytes (which may end in 0xff bytes, as a real stream's last word does).
// Candidates are all true field positions plus false ones: look-alikes 4 and 8 bytes in front of a
// true entry, look-alikes in the middle of a payload, positions inside a long delta.  Their context
// (terminator byte, 0xff run in front of it) is read from the image bytes, as the device does; a
// true candidate ends where its entry ends, a false one anywhere.  keep[] follows the product's rule
// (not within 13 bytes of a later candidate) with random extra drops and random extra keeps.
//
// Checked on every image:
//   1. dx_chain_walk finds exactly the true entries and their wells whenever every true candidate
//      decoded (stat == 0) -- whatever the false candidates look like;
//   2. (there is a kept candidate and all of them pass dx_chain_check_one)  <=>  (the walk succeeds and
//      reports as_assumed);
//   3. when as_assumed holds, the wells the layout assumed (first delta 255*ffrun + d, later ones d)
//      are the walk's wells;
//   4. the walk cut into windows at random bounds, each window starting at the cursor the one before
//      stopped at and carrying the last well (as the pipelined host decode walks): every window stops
//      at the first entry that starts at or past its bound, and together they find the same entries and
//      wells as the whole walk and end at n -- or, when the whole walk fails, a window fails.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include <algorithm>
#include "dx_chain.h"

static uint64_t rng_state = 0x9e3779b97f4a7c15ull;
static uint32_t rnd()
{ rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17;
  return (uint32_t) (rng_state >> 32);
}
static uint32_t rnd(uint32_t n) { return n ? rnd() % n : 0; }

struct Cand { int64_t q; int64_t end; int32_t stat; bool truth; int32_t well; };

int main(int argc, char **argv)
{ const int rounds = (argc > 1) ? atoi(argv[1]) : 20000;
  long assumed = 0, broken = 0, walked = 0, windowed = 0;
  for (int round = 0; round < rounds; round++)
    { rng_state += 0x632be59bd9b4e019ull * (uint64_t) (round + 1);
      const int style = (int) rnd(4);                  // 0: tidy files, 3: everything at once
      std::vector<uint8_t> img;
      const int64_t first = 2 + (int64_t) rnd(40);
      for (int64_t k = 0; k < first; k++) img.push_back((uint8_t) rnd(256));
      const int nent = 1 + (int) rnd(12);
      std::vector<Cand> cs;
      int32_t well = (int32_t) rnd(1000), well_in = well;
      for (int e = 0; e < nent; e++)
        { // delta: mostly small; sometimes >= 255 (0xff bytes), more often so for the first entry
          uint32_t delta = rnd(40);
          if ((e == 0 && rnd(3) == 0) || (style >= 2 && rnd(6) == 0)) delta = 255 * (1 + rnd(4)) + rnd(255);
          for (uint32_t k = 0; k < delta / 255; k++) img.push_back(0xff);
          img.push_back((uint8_t) (delta % 255));
          well += (int32_t) delta;
          Cand c; c.q = (int64_t) img.size(); c.truth = true; c.well = well;
          c.stat = (style == 3 && rnd(25) == 0) ? 1 : 0;
          for (int k = 0; k < 12; k++) img.push_back((uint8_t) rnd(256));
          const int plen = 4 * (int) (1 + rnd(30));
          for (int k = 0; k < plen; k++) img.push_back((uint8_t) rnd(256));
          // the payload's tail: zero padding, or 0xff bytes (one stream in 200 ends in one)
          const int tail = (int) rnd(4);
          const uint32_t how = rnd(style == 0 ? 2 : 4);
          for (int k = 0; k < tail; k++) img[img.size() - 1 - (size_t) k] = (how == 3) ? 0xff : (how == 2 ? (uint8_t) rnd(256) : 0);
          c.end = (int64_t) img.size();
          cs.push_back(c);
        }
      const int64_t n = (int64_t) img.size();
      // false candidates
      const int ntrue = (int) cs.size();
      for (int e = 0; e < ntrue && style >= 1; e++)
        { for (int d = 4; d <= 8; d += 4)
            if (rnd(3) == 0 && cs[e].q - d > first + 1)
              { Cand f; f.q = cs[e].q - d; f.truth = false; f.well = 0;
                f.stat = (int32_t) (rnd(3) != 0);
                f.end = f.q + 12 + (int64_t) rnd(200);
                if (rnd(4) == 0) f.end = cs[e].end;
                cs.push_back(f);
              }
          if (rnd(4) == 0)                                        // a look-alike inside the payload (or the delta)
            { Cand f; f.q = cs[e].q + 1 + (int64_t) rnd((uint32_t) (cs[e].end - cs[e].q - 1)); f.truth = false; f.well = 0;
              f.stat = (int32_t) (rnd(2) != 0);
              f.end = f.q + 12 + (int64_t) rnd(300);
              if (f.q + 12 <= n) cs.push_back(f);
            }
          if (style == 3 && rnd(4) == 0 && cs[e].q - 2 > first + 1)    // inside the delta bytes / the previous tail
            { Cand f; f.q = cs[e].q - 1 - (int64_t) rnd(3); f.truth = false; f.well = 0;
              f.stat = (int32_t) (rnd(2) != 0);
              f.end = (rnd(2) == 0) ? cs[e].end : f.q + 12 + (int64_t) rnd(100);
              cs.push_back(f);
            }
        }
      std::sort(cs.begin(),cs.end(),[](const Cand &a, const Cand &b) { return a.q < b.q; });
      cs.erase(std::unique(cs.begin(),cs.end(),[](const Cand &a, const Cand &b) { return a.q == b.q; }),cs.end());
      // (a duplicate position keeps the first of the two: make sure a true one survives)
      const int64_t N = (int64_t) cs.size();
      std::vector<int64_t> q(N), soff(6*N);
      std::vector<int32_t> ffrun(N), stat(N), rlen_d(N);
      std::vector<uint8_t> last(N), keep(N);
      int ntrue_left = 0;
      for (int64_t i = 0; i < N; i++)
        { q[i] = cs[i].q; stat[i] = cs[i].stat;
          if (cs[i].end > n) cs[i].end = n;
          for (int k = 0; k < 6; k++) soff[6*i + k] = cs[i].end;
          const int64_t p = q[i] - 1;
          last[i] = img[(size_t) p];
          int32_t r = 0;
          for (int64_t k = p - 1; k >= first && img[(size_t) k] == 0xff; k--) r++;
          ffrun[i] = r;
          rlen_d[i] = (stat[i] != 0 && rnd(2) == 0) ? -1 : 100;
          ntrue_left += cs[i].truth;
        }
      if (ntrue_left != ntrue) continue;                                   // a true entry lost to a duplicate
      for (int64_t i = 0; i < N; i++)
        { bool k = !(i + 1 < N && q[i+1] - q[i] < 13);
          if (style == 3 && rnd(30) == 0) k = !k;                           // the plausibility filter, either way
          keep[i] = k ? 1 : 0;
        }
      DxChainIn ci = { q.data(), ffrun.data(), last.data(), stat.data(), soff.data(), keep.data(), N, first, n };
      std::vector<int32_t> cand(N + 1), wells(N + 1);
      int64_t M = 0, stop = 0;
      bool as_assumed = false;
      const bool ok = dx_chain_walk(ci,well_in,cand.data(),wells.data(),&M,&as_assumed,&stop);
      if (ok && stop != n)
        { fprintf(stderr,"round %d: the walk stopped at %lld, image length %lld\n",round,(long long) stop,(long long) n); return 1; }

      // 1. the walk against the truth
      bool all_decoded = true;
      for (int64_t i = 0; i < N; i++) if (cs[i].truth && stat[i]) all_decoded = false;
      if (all_decoded)
        { if (!ok || M != ntrue)
            { fprintf(stderr,"round %d: walk ok %d, %lld entries, truth %d\n",round,(int) ok,(long long) M,ntrue); return 1; }
          int t = 0;
          for (int64_t i = 0; i < N; i++)
            if (cs[i].truth)
              { if (cand[t] != (int32_t) i || wells[t] != cs[i].well)
                  { fprintf(stderr,"round %d: entry %d is candidate %d (want %lld), well %d (want %d)\n",round,t,
                            cand[t],(long long) i,wells[t],cs[i].well); return 1; }
                t++;
              }
          walked++;
        }
      else if (!ok) broken++;

      // 2. the predicate form
      bool all_pass = true;
      int64_t nkept = 0;
      for (int64_t i = 0; i < N; i++)
        if (keep[i])
          { nkept++;
            if (!dx_chain_check_one(ci,rlen_d.data(),i)) all_pass = false;
          }
      if (nkept == 0) all_pass = false;                                   // nothing kept proves nothing
      // (rlen_d < 0 only where stat != 0, which fails both forms)
      if (all_pass != (ok && as_assumed))
        { fprintf(stderr,"round %d: predicate %d, walk %d, as assumed %d (N %lld, M %lld)\n",round,(int) all_pass,
                  (int) ok,(int) as_assumed,(long long) N,(long long) M); return 1; }

      // 3. the wells the layout assumed
      if (ok && as_assumed)
        { int64_t w = well_in; int t = 0;
          for (int64_t i = 0; i < N; i++)
            { if (!keep[i]) continue;
              const int64_t p = q[i] - 1;
              uint32_t delta = last[i];
              if (ffrun[i] > 0 && p - ffrun[i] == first) delta += 255u * (uint32_t) ffrun[i];
              w += delta;
              if (wells[t] != (int32_t) w)
                { fprintf(stderr,"round %d: assumed well %lld, walk %d at entry %d\n",round,(long long) w,wells[t],t); return 1; }
              t++;
            }
          assumed++;
        }

      // 4. window by window (the bounds are drawn without changing the images of the later rounds)
      { const uint64_t image_rng = rng_state;
        std::vector<int64_t> bounds;                                      // the windows' stops, the last one n
        const int nwin = 2 + (int) rnd(6);
        for (int w = 0; w + 1 < nwin; w++) bounds.push_back(first + (int64_t) rnd((uint32_t) (n - first)));
        std::sort(bounds.begin(),bounds.end());
        bounds.push_back(n);
        DxChainIn wi = ci;
        wi.keep = NULL;                                                   // the pipelined decode assumes no layout
        std::vector<int32_t> wc(N + 1), ww(N + 1), allc, allw;
        int32_t wwell = well_in;
        bool wok = true, dummy;
        int busy = 0;                                                     // windows with an entry (or the break)
        for (const int64_t b : bounds)
          { int64_t m = 0, cur = 0;
            wi.stop = b;
            if (!dx_chain_walk(wi,wwell,wc.data(),ww.data(),&m,&dummy,&cur)) { wok = false; busy++; break; }
            const int64_t last_start = (m > 1) ? soff[6*wc[m-2] + 5] : wi.start;    // where its last entry starts
            if (cur < b || (m > 0 && last_start >= b))
              { fprintf(stderr,"round %d: a window bounded by %lld stopped at %lld, its last entry starts at %lld\n",
                        round,(long long) b,(long long) cur,(long long) last_start); return 1; }
            if (m > 0) { wwell = ww[m-1]; busy++; }
            allc.insert(allc.end(),wc.begin(),wc.begin() + m);
            allw.insert(allw.end(),ww.begin(),ww.begin() + m);
            wi.start = cur;
          }
        if (wok != ok ||
            (ok && (wi.start != n || allc != std::vector<int32_t>(cand.begin(),cand.begin() + M) ||
                    allw != std::vector<int32_t>(wells.begin(),wells.begin() + M))))
          { fprintf(stderr,"round %d: windowed walk ok %d, whole walk ok %d (%zu windows, %zu / %lld entries)\n",round,
                    (int) wok,(int) ok,bounds.size(),allc.size(),(long long) M); return 1; }
        if (busy >= 2) windowed++;
        rng_state = image_rng;
      }
    }
  printf("ok %d images: %ld walked to the truth, %ld as assumed, %ld broken chains refused, %ld walked in windows\n",
         rounds,walked,assumed,broken,windowed);
  return 0;
}
