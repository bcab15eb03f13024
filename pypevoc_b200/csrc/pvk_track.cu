// pvk_track.cu -- partial tracking (PV.toSinSum -> SinSum.add_frame, PVAnalysis.py:299-322,
// 871-957) as a handful of small GPU kernels.
//
// The reference's greedy match of frame j against frame j-1 depends on those two peak rows
// only (SURVEY appendix A5), so tracking splits into
//   link     one warp per frame pair: peaks of frame j in descending magnitude each take the
//            nearest still-unused peak of frame j-1 (|17.312*(fc/fp-1)| < maxpitchjmp,
//            :914-928) or start a new partial (:941)
//   scan     exclusive scan of new-partial counts -> ids in add_empty_partial call order (:819-830)
//   resolve  continued peaks inherit the id of their predecessor: chunk-local propagation,
//            a short sequential pass over chunk boundaries, final fix-up
//   pack     per-track runs (= RegPartial.f/mag/ph/realph lists, :616-626) for resynthesis
// Exact magnitude ties inside one frame (measure zero for real signals) are ordered by column
// (current frame: higher column first, previous frame: lower column first); the reference's
// order there comes from numpy's unstable argsort and python's tuple sort on track index.
#include "pvk_common.cuh"
#include <stdlib.h>

namespace pvk {

constexpr int LINK_NONE = -1;    // slot is not a point
// link <= -2: new partial, rank among the frame's new partials = -2 - link

// ------------------------------------------------------------------ link
// abs(17.312*(fc/pf - 1.0)): dpitch2st :62-68 as called at :914
__device__ __forceinline__ double stonediff(double fc, double pfv) {
  return fabs(__dmul_rn(17.312, __dsub_rn(__ddiv_rn(fc, pfv), 1.0)));
}

// The reference's loop, one current peak at a time (:903-950); the whole warp scans the previous
// row for the nearest unused peak.  Works for any K <= 1024.  Returns the number of new partials.
__device__ __forceinline__ int link_greedy_generic(const double *cf, const double *pf, const double *pm,
                                                   const short *ord, const short *prank, int nc, int phi,
                                                   double maxjump, int32_t *__restrict__ link_row) {
  const int lane = threadIdx.x & 31;
  unsigned usedmask = 0;
  int nnew = 0;
  for (int t = 0; t < nc; ++t) {
    const int c = ord[t];
    const double fc = cf[c];
    double bd = 1e300;
    int br = 0x7fffffff, bp = -1;
    for (int p = lane, q = 0; p < phi; p += 32, ++q) {
      if (pm[p] > 0.0 && !((usedmask >> q) & 1u)) {
        const double d = stonediff(fc, pf[p]);
        const int r = prank[p];
        if (d < bd || (d == bd && r < br)) { bd = d; br = r; bp = p; }
      }
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
      const double od = __shfl_xor_sync(FULL, bd, o);
      const int orr = __shfl_xor_sync(FULL, br, o), op = __shfl_xor_sync(FULL, bp, o);
      if (od < bd || (od == bd && orr < br)) { bd = od; br = orr; bp = op; }
    }
    int lk;
    if (bp >= 0 && bd < maxjump) {                              // :923
      lk = bp;
      if ((bp & 31) == lane) usedmask |= 1u << (bp >> 5);
    } else {
      lk = -2 - nnew;                                           // add_empty_partial :941
      ++nnew;
    }
    if (lane == 0) link_row[c] = lk;
  }
  return nnew;
}

// ---- large rows (K > 128): ranks by a warp bitonic sort, nearest-unused search inside a window
// Sort (magnitude, column) pairs of one row held in shared memory: descending magnitude, ties by
// column (hi_first: higher column first -- the current row's rule; else lower column first --
// the previous row's).  KP = power of two >= the row length; invalid slots carry magnitude -1
// and end up last.  O(KP log^2 KP / 32) per lane instead of the O(K^2 / 32) counting rank.
__device__ __forceinline__ void warp_sort_desc(double *key, short *idx, int KP, bool hi_first) {
  const int lane = threadIdx.x & 31;
  for (int k = 2; k <= KP; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = lane; i < KP; i += 32) {
        const int x = i ^ j;
        if (x > i) {
          const double a = key[i], b = key[x];
          const short ia = idx[i], ib = idx[x];
          // "a sorts before b"
          const bool a_first = a > b || (a == b && (hi_first ? ia > ib : ia < ib));
          const bool up = (i & k) == 0;
          if (up ? !a_first : a_first) { key[i] = b; key[x] = a; idx[i] = ib; idx[x] = ia; }
        }
      }
      __syncwarp();
    }
  }
}

// The reference's loop (:903-950) for one row, one current peak at a time; when the previous
// row is a gap-free ascending run of frequencies (rows come out of the analysis in bin order)
// only the window of previous peaks that can lie within maxpitchjmp is scanned: it is found by a
// binary search on the fp32 frequencies with the fast kernel's guard band, every peak outside it
// has a distance >= maxjump and can never be taken (:923).  Returns the number of new partials.
__device__ __forceinline__ int link_greedy_window(const double *cf, const double *pf, const float *pf32,
                                                  const short *ord, const short *prank, unsigned *usedw,
                                                  int nc, int phi, int KP, double maxjump, float eps32,
                                                  int32_t *__restrict__ link_row) {
  const int lane = threadIdx.x & 31;
  for (int w = lane; w < (phi + 31) / 32; w += 32) usedw[w] = 0u;
  __syncwarp();
  int nnew = 0;
  for (int t = 0; t < nc; ++t) {
    const int c = ord[t];
    const double fc = cf[c];
    const float fc32 = (float)fc;
    const float flo = fc32 * (1.f - eps32), fhi = fc32 * (1.f + eps32 + 2.f * eps32 * eps32);
    int p0 = 0;
    for (int step = KP >> 1; step >= 1; step >>= 1) {
      const int mid = p0 + step;
      if (mid <= phi && pf32[mid - 1] < flo) p0 = mid;
    }
    double bd = 1e300;
    int br = 0x7fffffff, bp = -1;
    for (int pb = p0; pb < phi; pb += 32) {
      if (pf32[pb] > fhi) break;                                  // warp uniform
      const int p = pb + lane;
      if (p < phi) {
        const float pv = pf32[p];
        if (fabsf(fc32 - pv) < eps32 * pv && !((usedw[p >> 5] >> (p & 31)) & 1u)) {
          const double d = stonediff(fc, pf[p]);
          const int r = prank[p];
          if (d < bd || (d == bd && r < br)) { bd = d; br = r; bp = p; }
        }
      }
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
      const double od = __shfl_xor_sync(FULL, bd, o);
      const int orr = __shfl_xor_sync(FULL, br, o), op = __shfl_xor_sync(FULL, bp, o);
      if (od < bd || (od == bd && orr < br)) { bd = od; br = orr; bp = op; }
    }
    int lk;
    if (bp >= 0 && bd < maxjump) {                              // :923
      lk = bp;
      if (lane == 0) usedw[bp >> 5] |= 1u << (bp & 31);
    } else {
      lk = -2 - nnew;                                           // add_empty_partial :941
      ++nnew;
    }
    if (lane == 0) link_row[c] = lk;
    __syncwarp();
  }
  return nnew;
}

__host__ __device__ constexpr int link_pow2(int K) {
  int p = 32;
  while (p < K) p <<= 1;
  return p;
}
// per warp: cf cm pf pm (double, K) | sort keys (double, KP) | pf32 (float, K) | usedw (32 words)
//           | ord prank (short, K) | sort columns (short, KP)
__host__ __device__ constexpr int link_generic_smem_per_warp(int K) {
  return (K * (4 * 8 + 4 + 2 * 2) + link_pow2(K) * (8 + 2) + 32 * 4 + 15) / 16 * 16;
}

__global__ void track_link_kernel(const double *__restrict__ f, const double *__restrict__ mag,
                                  int64_t nrows, int64_t F, int K, double maxjump,
                                  int32_t *__restrict__ link, int32_t *__restrict__ newcount) {
  PVK_SMEM(smem);
  const int W = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KP = link_pow2(K);
  unsigned char *base = smem + (size_t)warp * link_generic_smem_per_warp(K);
  double *cf = reinterpret_cast<double *>(base);
  double *cm = cf + K;
  double *pf = cm + K;
  double *pm = pf + K;
  double *skey = pm + K;
  float *pf32 = reinterpret_cast<float *>(skey + KP);
  unsigned *usedw = reinterpret_cast<unsigned *>(pf32 + K);
  short *ord = reinterpret_cast<short *>(usedw + 32);
  short *prank = ord + K;
  short *sidx = prank + K;
  const float eps32 = (float)(maxjump / 17.312 * (1.0 + 1e-4) + 1e-6);   // guard band as in the fast kernel
  for (int64_t row = (int64_t)blockIdx.x * W + warp; row < nrows; row += (int64_t)gridDim.x * W) {
    const bool has_prev = (row % F) > 0;
    // ---- load both rows (invalid slots: magnitude -1)
    int nc = 0, phi = 0;
    bool okasc = true;
    for (int i0 = 0; i0 < K; i0 += 32) {
      const int i = i0 + lane;
      bool v = false;
      if (i < K) {
        const double a = f[row * K + i], b = mag[row * K + i];
        v = a > 0.0 && b > 0.0;                                   // :876
        cf[i] = a; cm[i] = v ? b : -1.0;
        if (!v) link[row * K + i] = LINK_NONE;
        if (has_prev) {
          const double c = f[(row - 1) * K + i], d = mag[(row - 1) * K + i];
          const bool vp = c > 0.0 && d > 0.0;
          pf[i] = c; pm[i] = vp ? d : -1.0;
          pf32[i] = vp ? (float)c : -1.f;
          if (vp) phi = i + 1;
        }
      }
      nc += __popc(__ballot_sync(FULL, v));
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) phi = max(phi, __shfl_xor_sync(FULL, phi, o));
    __syncwarp();
    // ---- order of the current peaks: magnitude descending (:874-875), ties higher column first
    for (int i = lane; i < KP; i += 32) { skey[i] = i < K ? cm[i] : -1.0; sidx[i] = (short)i; }
    __syncwarp();
    warp_sort_desc(skey, sidx, KP, true);
    for (int t = lane; t < nc; t += 32) ord[t] = sidx[t];
    __syncwarp();
    int nnew;
    if (!has_prev || phi == 0) {
      for (int t = lane; t < nc; t += 32) link[row * K + ord[t]] = -2 - t;   // everything is new (:941)
      nnew = nc;
    } else {
      // ---- rank of the previous peaks in descending magnitude (:891-900), ties lower column first
      for (int i = lane; i < KP; i += 32) { skey[i] = i < phi ? pm[i] : -1.0; sidx[i] = (short)i; }
      __syncwarp();
      warp_sort_desc(skey, sidx, KP, false);
      for (int t = lane; t < KP; t += 32) {
        const int i = sidx[t];
        if (i < phi) prank[i] = (short)(skey[t] > 0.0 ? t : 0);
      }
      for (int p = lane; p < phi; p += 32)
        okasc = okasc && pm[p] > 0.0 && (p + 1 >= phi || (pm[p + 1] > 0.0 && pf32[p] <= pf32[p + 1]));
      const bool asc = __all_sync(FULL, okasc);
      __syncwarp();
      nnew = asc ? link_greedy_window(cf, pf, pf32, ord, prank, usedw, nc, phi, KP, maxjump, eps32, link + row * K)
                 : link_greedy_generic(cf, pf, pm, ord, prank, nc, phi, maxjump, link + row * K);
    }
    if (lane == 0) newcount[row] = nnew;
    __syncwarp();
  }
}

// ---- rows of up to 128 peaks: the greedy loop without ranking either row.
// The sequential loop (:903-950) hands every current peak, in descending magnitude order, its
// nearest still-unused previous peak (if within maxpitchjmp).  Only peaks that compete for the same
// previous peak need to know who comes first, and that is a direct magnitude comparison:
//   * lane owns the current peaks in COLUMNS lane + 32 s; the previous peaks within maxpitchjmp of
//     one (exact fp64 distance) form a bit mask over a window of <= 32 consecutive columns that
//     starts at a binary-searched column (previous rows come out of the analysis in ascending
//     frequency order; other rows scan from column 0);
//   * a round: every unresolved peak proposes its nearest unused candidate (distance ties: larger
//     previous magnitude, then lower column = lower rank, :891-900,:914-922); a proposed previous
//     peak goes to the proposer that comes first in the order (atomicMax on the magnitude's bit
//     pattern, then on the column among equal magnitudes: ties -> higher column first, :874-875).
//     Everybody that comes before the EARLIEST LOSER keeps what it proposed (an earlier peak is
//     never affected by a later one, and losing somebody else's target does not change one's own
//     arg-min); the loser and everybody after it try again; a peak without unused candidates is a
//     new partial.  "Before the loser" is a magnitude comparison with the loser.  Conflict-free rows
//     finish in one round.
//   * new partials are numbered by descending magnitude among themselves (:941).
// Same result as the loop, bit for bit (tests/fuzz_emu.py).  Rows with a window wider than 32
// columns (previous row with holes / out of order and more than 32 columns) take the loop itself.
__host__ __device__ constexpr int link_claim_smem_per_warp(int S) {
  // cf cm pf pm (double) | claim magnitudes = sort keys (8) | pf32 (4) | claim columns (4) | ord prank sidx (short) | usedw
  return 32 * S * (4 * 8 + 8 + 4 + 4 + 3 * 2) + 3 * 32 * 4;
}

template <int S>
__global__ void track_link_claim_kernel(const double *__restrict__ f, const double *__restrict__ mag,
                                        int64_t nrows, int64_t F, int K, double maxjump,
                                        int32_t *__restrict__ link, int32_t *__restrict__ newcount) {
  PVK_SMEM(smem);
  constexpr int KM = 32 * S;
  const int W = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char *base = smem + (size_t)warp * link_claim_smem_per_warp(S);
  double *cf = reinterpret_cast<double *>(base);
  double *cm = cf + KM;
  double *pf = cm + KM;
  double *pm = pf + KM;
  unsigned long long *claim_m = reinterpret_cast<unsigned long long *>(pm + KM);   // [KM]; the loop's sort keys too
  float *pf32 = reinterpret_cast<float *>(claim_m + KM);          // [KM] previous frequencies, -1 = not a point
  int *claim_c = reinterpret_cast<int *>(pf32 + KM);              // [KM]
  short *ord = reinterpret_cast<short *>(claim_c + KM);
  short *prank = ord + KM;
  short *sidx = prank + KM;
  unsigned *usedw = reinterpret_cast<unsigned *>(sidx + KM);      // [32]
  unsigned *propw = usedw + 32, *confw = propw + 32;              // [32] each
  for (int p = lane; p < KM; p += 32) { claim_m[p] = 0ull; claim_c[p] = -1; }
  // fp32 pre-test window: |fc - fp| < eps32 * fp is implied by |17.312 (fc/fp - 1)| < maxjump
  // (slack 1e-4 relative + 1e-6 absolute >> fp32 rounding of fc and fp); the exact fp64 test decides
  const float eps32 = (float)(maxjump / 17.312 * (1.0 + 1e-4) + 1e-6);

  for (int64_t row = (int64_t)blockIdx.x * W + warp; row < nrows; row += (int64_t)gridDim.x * W) {
    const bool has_prev = (row % F) > 0;
    int32_t *lrow = link + row * K;
    int phi = 0;
    double mine[S], fmine[S];
#pragma unroll
    for (int s = 0; s < S; ++s) {
      const int i = lane + 32 * s;
      double cmv = -1.0, pmv = -1.0, cfv = 0.0;
      float p32 = -1.f;
      if (i < K) {
        const double a = f[row * K + i], b = mag[row * K + i];
        const bool v = a > 0.0 && b > 0.0;                        // :876
        cfv = a; cmv = v ? b : -1.0;
        if (!v) lrow[i] = LINK_NONE;
        if (has_prev) {
          const double c = f[(row - 1) * K + i], d = mag[(row - 1) * K + i];
          const bool vp = c > 0.0 && d > 0.0;
          pf[i] = c; pmv = vp ? d : -1.0;
          p32 = vp ? (float)c : -1.f;
          if (vp) phi = i + 1;
        }
      }
      cf[i] = cfv; cm[i] = cmv; pm[i] = pmv; pf32[i] = p32;
      mine[s] = cmv; fmine[s] = cfv;
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) phi = max(phi, __shfl_xor_sync(FULL, phi, o));
    usedw[lane] = 0u;
    __syncwarp();
    bool okasc = true;
    for (int p = lane; p < phi; p += 32)
      okasc = okasc && pm[p] > 0.0 && (p + 1 >= phi || (pm[p + 1] > 0.0 && pf32[p] <= pf32[p + 1]));
    const bool asc = __all_sync(FULL, okasc);

    // ---- candidate masks: bit b of cmask[s] = previous column p0[s] + b is within maxpitchjmp
    int p0[S], res[S], prop[S];                                   // res: -3 unresolved, -2 new, -4 no peak, >= 0 matched column
    unsigned cmask[S];
    bool overflow = false;
#pragma unroll
    for (int s = 0; s < S; ++s) {
      p0[s] = 0; cmask[s] = 0u; prop[s] = -1;
      res[s] = mine[s] > 0.0 ? -3 : -4;
      if (mine[s] > 0.0 && phi > 0) {
        const double fc = fmine[s];
        const float fc32 = (float)fc;
        float fhi = 3.0e38f;
        int q = 0;
        if (asc) {
          // every p passing the window test below has pf32[p] in [flo, fhi]
          const float flo = fc32 * (1.f - eps32);
          fhi = fc32 * (1.f + eps32 + 2.f * eps32 * eps32);
#pragma unroll
          for (int step = KM / 2; step >= 1; step >>= 1) {
            const int mid = q + step;
            if (mid <= phi && pf32[mid - 1] < flo) q = mid;
          }
        }
        p0[s] = q;
        // the first proposal falls out of the same pass: nearest candidate; distance ties: larger previous
        // magnitude, then lower column (ascending scan + strict comparisons)
        double bd = 1e300, bm = -1.0;
        for (int p = q; p < phi; ++p) {
          const float pv = pf32[p];
          if (pv > fhi) break;
          if (fabsf(fc32 - pv) < eps32 * pv) {
            const double d = stonediff(fc, pf[p]);
            if (d < maxjump) {                                    // :923: only these can ever match
              if (p - q < 32) cmask[s] |= 1u << (p - q); else overflow = true;
              const double m = pm[p];
              if (d < bd || (d == bd && m > bm)) { bd = d; bm = m; prop[s] = p; }
            }
          }
        }
      }
    }
    if (__any_sync(FULL, overflow)) {
      // ---- rare: the reference's loop itself, with both rows ranked by a warp bitonic sort
      double *skey = reinterpret_cast<double *>(claim_m);
      int nc = 0;
#pragma unroll
      for (int s = 0; s < S; ++s) nc += __popc(__ballot_sync(FULL, mine[s] > 0.0));
      for (int i = lane; i < KM; i += 32) { skey[i] = cm[i]; sidx[i] = (short)i; }
      __syncwarp();
      warp_sort_desc(skey, sidx, KM, true);
      for (int t = lane; t < nc; t += 32) ord[t] = sidx[t];
      __syncwarp();
      for (int i = lane; i < KM; i += 32) { skey[i] = i < phi ? pm[i] : -1.0; sidx[i] = (short)i; }
      __syncwarp();
      warp_sort_desc(skey, sidx, KM, false);
      for (int t = lane; t < KM; t += 32) {
        const int i = sidx[t];
        if (i < phi) prank[i] = (short)(skey[t] > 0.0 ? t : 0);
      }
      __syncwarp();
      const int nnew = link_greedy_generic(cf, pf, pm, ord, prank, nc, phi, maxjump, lrow);
      if (lane == 0) newcount[row] = nnew;
      __syncwarp();
      for (int p = lane; p < KM; p += 32) claim_m[p] = 0ull;      // (was the sort's key array)
      __syncwarp();
      continue;
    }

    // ---- propose / commit rounds.  propw / confw: previous columns proposed / proposed more than once
    //      in this round; claim_m / claim_c are only touched for contested columns and are reset by
    //      their users (all-zero / -1 between rounds and rows)
    for (;;) {
      bool pend = false;
#pragma unroll
      for (int s = 0; s < S; ++s) pend = pend || (res[s] == -3 && cmask[s] != 0u);
      if (!__any_sync(FULL, pend)) break;
      propw[lane] = 0u; confw[lane] = 0u;
      __syncwarp();
      bool act[S];
      bool clash = false;
#pragma unroll
      for (int s = 0; s < S; ++s) {
        act[s] = false;
        if (res[s] == -3 && cmask[s] != 0u) {
          // a kept proposal stays the arg-min while its target is unused (the unused set only shrinks)
          if (prop[s] < 0 || ((usedw[prop[s] >> 5] >> (prop[s] & 31)) & 1u)) {
            // nearest unused candidate; distance ties: larger previous magnitude, then lower column
            const double fc = fmine[s];
            double bd = 1e300, bm = -1.0;
            int bp = -1;
            for (unsigned rem = cmask[s]; rem; rem &= rem - 1u) {
              const int p = p0[s] + __ffs((int)rem) - 1;
              if ((usedw[p >> 5] >> (p & 31)) & 1u) { cmask[s] &= ~(rem & (0u - rem)); continue; }   // taken: drop it
              const double d = stonediff(fc, pf[p]);
              const double m = pm[p];
              if (d < bd || (d == bd && m > bm)) { bd = d; bm = m; bp = p; }
            }
            prop[s] = bp;
          }
          if (prop[s] >= 0) {
            act[s] = true;
            const unsigned bit = 1u << (prop[s] & 31);
            if (atomicOr(&propw[prop[s] >> 5], bit) & bit) { atomicOr(&confw[prop[s] >> 5], bit); clash = true; }
          }
        }
      }
      __syncwarp();
      if (!__any_sync(FULL, clash)) {
        // nobody shares a target: every proposal stands, whatever the order
#pragma unroll
        for (int s = 0; s < S; ++s) if (act[s]) res[s] = prop[s];
        __syncwarp();
        usedw[lane] |= propw[lane];
        __syncwarp();
        continue;
      }
      // contested targets go to the proposer that comes first in the order: magnitude, then column
      bool cont[S];
#pragma unroll
      for (int s = 0; s < S; ++s) {
        cont[s] = act[s] && ((confw[prop[s] >> 5] >> (prop[s] & 31)) & 1u);
        if (cont[s]) atomicMax(&claim_m[prop[s]], (unsigned long long)__double_as_longlong(mine[s]));
      }
      __syncwarp();
#pragma unroll
      for (int s = 0; s < S; ++s) {
        if (cont[s] && claim_m[prop[s]] == (unsigned long long)__double_as_longlong(mine[s]))
          atomicMax(&claim_c[prop[s]], lane + 32 * s);
      }
      __syncwarp();
      // the earliest loser in the order (magnitude descending, ties higher column first): everybody
      // before it keeps what it proposed, the loser and everybody after it try again
      unsigned long long lk = 0ull;
      int lc = -1;
      bool win[S];
#pragma unroll
      for (int s = 0; s < S; ++s) {
        const unsigned long long key = (unsigned long long)__double_as_longlong(mine[s]);
        win[s] = act[s] && (!cont[s] || (claim_m[prop[s]] == key && claim_c[prop[s]] == lane + 32 * s));
        if (act[s] && !win[s] && (key > lk || (key == lk && lane + 32 * s > lc))) { lk = key; lc = lane + 32 * s; }
      }
      __syncwarp();
#pragma unroll
      for (int s = 0; s < S; ++s) if (cont[s]) { claim_m[prop[s]] = 0ull; claim_c[prop[s]] = -1; }   // (all users write the same)
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) {
        const unsigned long long ok = __shfl_xor_sync(FULL, lk, o);
        const int oc = __shfl_xor_sync(FULL, lc, o);
        if (ok > lk || (ok == lk && oc > lc)) { lk = ok; lc = oc; }
      }
#pragma unroll
      for (int s = 0; s < S; ++s) {
        if (win[s]) {
          const unsigned long long key = (unsigned long long)__double_as_longlong(mine[s]);
          if (key > lk || (key == lk && lane + 32 * s > lc)) {
            res[s] = prop[s];
            atomicOr(&usedw[prop[s] >> 5], 1u << (prop[s] & 31));
          }
        }
      }
      __syncwarp();
    }
    // ---- links; new partials numbered by descending magnitude, ties higher column first (:874-875, :941)
    unsigned newm[S];
    int nnew = 0;
#pragma unroll
    for (int s = 0; s < S; ++s) { newm[s] = __ballot_sync(FULL, res[s] == -3); nnew += __popc(newm[s]); }
    int rk[S];
#pragma unroll
    for (int s = 0; s < S; ++s) rk[s] = 0;
    if (nnew > 1) {
#pragma unroll
      for (int s2 = 0; s2 < S; ++s2) {
        for (unsigned rem = newm[s2]; rem; rem &= rem - 1u) {
          const int c2 = 32 * s2 + __ffs((int)rem) - 1;
          const double m2 = cm[c2];
#pragma unroll
          for (int s = 0; s < S; ++s) rk[s] += (m2 > mine[s] || (m2 == mine[s] && c2 > lane + 32 * s)) ? 1 : 0;
        }
      }
    }
#pragma unroll
    for (int s = 0; s < S; ++s) {
      if (res[s] >= 0) lrow[lane + 32 * s] = res[s];
      else if (res[s] == -3) lrow[lane + 32 * s] = -2 - rk[s];
    }
    if (lane == 0) newcount[row] = nnew;
    __syncwarp();
  }
}

// ---- wide rows (K > 128): the same rank-free schedule with one CTA per frame pair.  A row of a few
// hundred peaks on ONE warp is a long serial chain (16 slots per lane, a dozen rounds on dense rows);
// spread over T = 128 / 256 threads with two columns each, a row takes 1/4 - 1/8 of the time, which is
// what matters when there are few rows (60 s at hop 1024 are 2 800 rows for 148 SMs).  Thread t owns
// columns t and t + T; warp collectives become block barriers / counts, the earliest loser is reduced
// through shared memory.  Same result as track_link_claim_kernel and the loop, bit for bit.
__host__ __device__ constexpr int link_cta_smem(int KM) {
  // cf cm pf pm (double) | claim magnitudes = sort keys (8) | pf32 (4) | claim columns (4) | ord prank sidx (short)
  // | usedw propw confw newbits (KM/32 words each) | 32 loser keys + 32 loser columns + 4 ints
  return KM * (4 * 8 + 8 + 4 + 4 + 3 * 2) + 4 * (KM / 32) * 4 + 32 * 8 + 32 * 4 + 16;
}

__global__ void __launch_bounds__(256) track_link_cta_kernel(const double *__restrict__ f, const double *__restrict__ mag,
                                                             int64_t nrows, int64_t F, int K, double maxjump,
                                                             int32_t *__restrict__ link, int32_t *__restrict__ newcount) {
  PVK_SMEM(smem);
  constexpr int S = 2;
  const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, NW = T >> 5;
  const int KM = T * S, NWORD = KM / 32;
  double *cf = reinterpret_cast<double *>(smem);
  double *cm = cf + KM;
  double *pf = cm + KM;
  double *pm = pf + KM;
  unsigned long long *claim_m = reinterpret_cast<unsigned long long *>(pm + KM);
  unsigned long long *redk = claim_m + KM;                        // [32]
  float *pf32 = reinterpret_cast<float *>(redk + 32);
  int *claim_c = reinterpret_cast<int *>(pf32 + KM);
  int *redc = claim_c + KM;                                       // [32]
  int *bc = redc + 32;                                            // [4]
  unsigned *usedw = reinterpret_cast<unsigned *>(bc + 4);
  unsigned *propw = usedw + NWORD, *confw = propw + NWORD, *newbits = confw + NWORD;
  short *ord = reinterpret_cast<short *>(newbits + NWORD);
  short *prank = ord + KM;
  short *sidx = prank + KM;
  for (int p = tid; p < KM; p += T) { claim_m[p] = 0ull; claim_c[p] = -1; }
  const float eps32 = (float)(maxjump / 17.312 * (1.0 + 1e-4) + 1e-6);   // guard band as in the warp kernel

  for (int64_t row = blockIdx.x; row < nrows; row += gridDim.x) {
    const bool has_prev = (row % F) > 0;
    int32_t *lrow = link + row * K;
    if (tid == 0) bc[0] = 0;
    for (int w = tid; w < NWORD; w += T) usedw[w] = 0u;
    __syncthreads();
    int phil = 0;
    double mine[S], fmine[S];
#pragma unroll
    for (int s = 0; s < S; ++s) {
      const int i = tid + T * s;
      double cmv = -1.0, pmv = -1.0, cfv = 0.0, pfv = 0.0;
      float p32 = -1.f;
      if (i < K) {
        const double a = f[row * K + i], b = mag[row * K + i];
        const bool v = a > 0.0 && b > 0.0;                        // :876
        cfv = a; cmv = v ? b : -1.0;
        if (!v) lrow[i] = LINK_NONE;
        if (has_prev) {
          const double c = f[(row - 1) * K + i], d = mag[(row - 1) * K + i];
          const bool vp = c > 0.0 && d > 0.0;
          pfv = c; pmv = vp ? d : -1.0;
          p32 = vp ? (float)c : -1.f;
          if (vp) phil = i + 1;
        }
      }
      cf[i] = cfv; cm[i] = cmv; pf[i] = pfv; pm[i] = pmv; pf32[i] = p32;
      mine[s] = cmv; fmine[s] = cfv;
    }
    if (phil > 0) atomicMax(&bc[0], phil);
    __syncthreads();
    const int phi = bc[0];
    bool okasc = true;
    for (int p = tid; p < phi; p += T)
      okasc = okasc && pm[p] > 0.0 && (p + 1 >= phi || (pm[p + 1] > 0.0 && pf32[p] <= pf32[p + 1]));
    const bool asc = __syncthreads_count(okasc ? 0 : 1) == 0;

    // ---- candidate masks (as in track_link_claim_kernel)
    int p0[S], res[S], prop[S];
    unsigned cmask[S];
    bool overflow = false;
#pragma unroll
    for (int s = 0; s < S; ++s) {
      p0[s] = 0; cmask[s] = 0u; prop[s] = -1;
      res[s] = mine[s] > 0.0 ? -3 : -4;
      if (mine[s] > 0.0 && phi > 0) {
        const double fc = fmine[s];
        const float fc32 = (float)fc;
        float fhi = 3.0e38f;
        int q = 0;
        if (asc) {
          const float flo = fc32 * (1.f - eps32);
          fhi = fc32 * (1.f + eps32 + 2.f * eps32 * eps32);
          for (int step = KM / 2; step >= 1; step >>= 1) {
            const int mid = q + step;
            if (mid <= phi && pf32[mid - 1] < flo) q = mid;
          }
        }
        p0[s] = q;
        double bd = 1e300, bm = -1.0;                             // (the first proposal falls out of the same pass)
        for (int p = q; p < phi; ++p) {
          const float pv = pf32[p];
          if (pv > fhi) break;
          if (fabsf(fc32 - pv) < eps32 * pv) {
            const double d = stonediff(fc, pf[p]);
            if (d < maxjump) {                                    // :923
              if (p - q < 32) cmask[s] |= 1u << (p - q); else overflow = true;
              const double m = pm[p];
              if (d < bd || (d == bd && m > bm)) { bd = d; bm = m; prop[s] = p; }
            }
          }
        }
      }
    }
    if (__syncthreads_count(overflow ? 1 : 0) != 0) {
      // ---- rare: the reference's loop itself, run by warp 0 with both rows ranked by a bitonic sort
      if (warp == 0) {
        double *skey = reinterpret_cast<double *>(claim_m);
        int nc = 0;
        for (int i0 = 0; i0 < KM; i0 += 32) nc += __popc(__ballot_sync(FULL, cm[i0 + lane] > 0.0));
        for (int i = lane; i < KM; i += 32) { skey[i] = cm[i]; sidx[i] = (short)i; }
        __syncwarp();
        warp_sort_desc(skey, sidx, KM, true);
        for (int t = lane; t < nc; t += 32) ord[t] = sidx[t];
        __syncwarp();
        for (int i = lane; i < KM; i += 32) { skey[i] = i < phi ? pm[i] : -1.0; sidx[i] = (short)i; }
        __syncwarp();
        warp_sort_desc(skey, sidx, KM, false);
        for (int t = lane; t < KM; t += 32) {
          const int i = sidx[t];
          if (i < phi) prank[i] = (short)(skey[t] > 0.0 ? t : 0);
        }
        __syncwarp();
        const int nnew = link_greedy_generic(cf, pf, pm, ord, prank, nc, phi, maxjump, lrow);
        if (lane == 0) newcount[row] = nnew;
      }
      __syncthreads();
      for (int p = tid; p < KM; p += T) claim_m[p] = 0ull;        // (was the sort's key array)
      __syncthreads();
      continue;
    }

    // ---- propose / commit rounds
    for (;;) {
      bool pend = false;
#pragma unroll
      for (int s = 0; s < S; ++s) pend = pend || (res[s] == -3 && cmask[s] != 0u);
      if (__syncthreads_count(pend ? 1 : 0) == 0) break;
      for (int w = tid; w < NWORD; w += T) { propw[w] = 0u; confw[w] = 0u; }
      __syncthreads();
      bool act[S];
      bool clash = false;
#pragma unroll
      for (int s = 0; s < S; ++s) {
        act[s] = false;
        if (res[s] == -3 && cmask[s] != 0u) {
          if (prop[s] < 0 || ((usedw[prop[s] >> 5] >> (prop[s] & 31)) & 1u)) {
            const double fc = fmine[s];
            double bd = 1e300, bm = -1.0;
            int bp = -1;
            for (unsigned rem = cmask[s]; rem; rem &= rem - 1u) {
              const int p = p0[s] + __ffs((int)rem) - 1;
              if ((usedw[p >> 5] >> (p & 31)) & 1u) { cmask[s] &= ~(rem & (0u - rem)); continue; }
              const double d = stonediff(fc, pf[p]);
              const double m = pm[p];
              if (d < bd || (d == bd && m > bm)) { bd = d; bm = m; bp = p; }
            }
            prop[s] = bp;
          }
          if (prop[s] >= 0) {
            act[s] = true;
            const unsigned bit = 1u << (prop[s] & 31);
            if (atomicOr(&propw[prop[s] >> 5], bit) & bit) { atomicOr(&confw[prop[s] >> 5], bit); clash = true; }
          }
        }
      }
      if (__syncthreads_count(clash ? 1 : 0) == 0) {
#pragma unroll
        for (int s = 0; s < S; ++s) if (act[s]) res[s] = prop[s];
        for (int w = tid; w < NWORD; w += T) usedw[w] |= propw[w];
        __syncthreads();
        continue;
      }
      bool cont[S];
#pragma unroll
      for (int s = 0; s < S; ++s) {
        cont[s] = act[s] && ((confw[prop[s] >> 5] >> (prop[s] & 31)) & 1u);
        if (cont[s]) atomicMax(&claim_m[prop[s]], (unsigned long long)__double_as_longlong(mine[s]));
      }
      __syncthreads();
#pragma unroll
      for (int s = 0; s < S; ++s) {
        if (cont[s] && claim_m[prop[s]] == (unsigned long long)__double_as_longlong(mine[s]))
          atomicMax(&claim_c[prop[s]], tid + T * s);
      }
      __syncthreads();
      unsigned long long lk = 0ull;
      int lc = -1;
      bool win[S];
#pragma unroll
      for (int s = 0; s < S; ++s) {
        const unsigned long long key = (unsigned long long)__double_as_longlong(mine[s]);
        win[s] = act[s] && (!cont[s] || (claim_m[prop[s]] == key && claim_c[prop[s]] == tid + T * s));
        if (act[s] && !win[s] && (key > lk || (key == lk && tid + T * s > lc))) { lk = key; lc = tid + T * s; }
      }
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) {
        const unsigned long long ok = __shfl_xor_sync(FULL, lk, o);
        const int oc = __shfl_xor_sync(FULL, lc, o);
        if (ok > lk || (ok == lk && oc > lc)) { lk = ok; lc = oc; }
      }
      if (lane == 0) { redk[warp] = lk; redc[warp] = lc; }
      __syncthreads();                                            // (every claim has been read by now)
#pragma unroll
      for (int s = 0; s < S; ++s) if (cont[s]) { claim_m[prop[s]] = 0ull; claim_c[prop[s]] = -1; }
      lk = 0ull; lc = -1;
      for (int w = 0; w < NW; ++w) {
        const unsigned long long ok = redk[w];
        const int oc = redc[w];
        if (ok > lk || (ok == lk && oc > lc)) { lk = ok; lc = oc; }
      }
#pragma unroll
      for (int s = 0; s < S; ++s) {
        if (win[s]) {
          const unsigned long long key = (unsigned long long)__double_as_longlong(mine[s]);
          if (key > lk || (key == lk && tid + T * s > lc)) {
            res[s] = prop[s];
            atomicOr(&usedw[prop[s] >> 5], 1u << (prop[s] & 31));
          }
        }
      }
      __syncthreads();
    }
    // ---- links; new partials numbered by descending magnitude, ties higher column first (:874-875, :941)
#pragma unroll
    for (int s = 0; s < S; ++s) {
      const unsigned m = __ballot_sync(FULL, res[s] == -3);
      if (lane == 0) newbits[NW * s + warp] = m;                  // columns 32 (NW s + warp) ... + 31
    }
    __syncthreads();
    int nnew = 0;
    for (int w = 0; w < NWORD; ++w) nnew += __popc(newbits[w]);
    int rk[S];
#pragma unroll
    for (int s = 0; s < S; ++s) rk[s] = 0;
    if (nnew > 1) {
      for (int w = 0; w < NWORD; ++w) {
        for (unsigned rem = newbits[w]; rem; rem &= rem - 1u) {
          const int c2 = 32 * w + __ffs((int)rem) - 1;
          const double m2 = cm[c2];
#pragma unroll
          for (int s = 0; s < S; ++s) rk[s] += (m2 > mine[s] || (m2 == mine[s] && c2 > tid + T * s)) ? 1 : 0;
        }
      }
    }
#pragma unroll
    for (int s = 0; s < S; ++s) {
      if (res[s] >= 0) lrow[tid + T * s] = res[s];
      else if (res[s] == -3) lrow[tid + T * s] = -2 - rk[s];
    }
    if (tid == 0) newcount[row] = nnew;
    __syncthreads();
  }
}

// ------------------------------------------------------------------ exclusive scans
// Tiled exclusive scan of int32 counts in two launches, every CTA independent: (1) per-tile sums,
// (2) each tile adds up the sums of the tiles before it (a few hundred values even for an 8 hour
// signal), scans its own SCAN_TILE elements and writes them.  grid = (tiles, rows of `in`); the
// element count of a row is n, or min(n, *n_dev) when the count lives on the device.
constexpr int SCAN_BD = 256, SCAN_E = 16, SCAN_TILE = SCAN_BD * SCAN_E, SCAN_SMEM = 2 * (SCAN_BD / 32) * 8;

__device__ __forceinline__ int64_t scan_count(int64_t n, const int32_t *n_dev) {
  if (n_dev) { const int64_t m = *n_dev; return m < n ? m : n; }
  return n;
}

__device__ __forceinline__ void scan_load_tile(const int32_t *__restrict__ in, int64_t i0, int64_t n, int *v) {
  if (i0 + SCAN_E <= n && ((reinterpret_cast<uintptr_t>(in + i0) & 15) == 0)) {
#pragma unroll
    for (int j = 0; j < SCAN_E / 4; ++j) {
      const int4 q = *reinterpret_cast<const int4 *>(in + i0 + 4 * j);
      v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w;
    }
  } else {
#pragma unroll
    for (int j = 0; j < SCAN_E; ++j) v[j] = (i0 + j < n) ? in[i0 + j] : 0;
  }
}

// block-wide sum of one long long per thread (SCAN_BD threads), result in every thread
__device__ __forceinline__ long long scan_block_sum(long long v, long long *sh) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  long long t = 0;
#pragma unroll
  for (int w = 0; w < SCAN_BD / 32; ++w) t += sh[w];
  __syncthreads();
  return t;
}

__global__ void __launch_bounds__(SCAN_BD) scan_tile_sums_kernel(const int32_t *__restrict__ in, int64_t stride, int64_t n,
                                                                 const int32_t *__restrict__ n_dev, int64_t ntiles,
                                                                 long long *__restrict__ tsum) {
  PVK_SMEM(smem);
  long long *sh = reinterpret_cast<long long *>(smem);
  n = scan_count(n, n_dev);
  const int64_t t = blockIdx.x, row = blockIdx.y;
  if (t * SCAN_TILE >= n) {                                    // beyond a device-side count: nothing to read
    if (threadIdx.x == 0) tsum[row * ntiles + t] = 0;
    return;
  }
  int v[SCAN_E];
  scan_load_tile(in + row * stride, t * SCAN_TILE + (int64_t)threadIdx.x * SCAN_E, n, v);
  long long loc = 0;
#pragma unroll
  for (int j = 0; j < SCAN_E; ++j) loc += v[j];
  const long long tot = scan_block_sum(loc, sh);
  if (threadIdx.x == 0) tsum[row * ntiles + t] = tot;
}

// out[i] = sum of in[0..i) (TO = int32 or int64); the grand total goes to total[row] (int32,
// optional) and, when out_total is set, to out[n] (the one-past-the-end offset).
template <class TO>
__global__ void __launch_bounds__(SCAN_BD) scan_tile_apply_kernel(const int32_t *__restrict__ in, int64_t stride, int64_t n,
                                                                  const int32_t *__restrict__ n_dev, int64_t ntiles,
                                                                  const long long *__restrict__ tsum, TO *__restrict__ out,
                                                                  int64_t out_stride, int32_t *__restrict__ total,
                                                                  int out_total) {
  PVK_SMEM(smem);
  long long *sh = reinterpret_cast<long long *>(smem);
  long long *wsum = sh + SCAN_BD / 32;
  n = scan_count(n, n_dev);
  const int64_t t = blockIdx.x, row = blockIdx.y;
  if (t * SCAN_TILE >= n && t != ntiles - 1) return;           // beyond a device-side count (the last tile writes the totals)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long *ts = tsum + row * ntiles;
  long long before = 0;
  const int64_t tlive = (n + SCAN_TILE - 1) / SCAN_TILE;      // tiles holding elements
  for (int64_t i = tid; i < (t < tlive ? t : tlive); i += SCAN_BD) before += ts[i];
  before = scan_block_sum(before, sh);
  const int64_t i0 = t * SCAN_TILE + (int64_t)tid * SCAN_E;
  int v[SCAN_E];
  scan_load_tile(in + row * stride, i0, n, v);
  long long loc = 0;
#pragma unroll
  for (int j = 0; j < SCAN_E; ++j) loc += v[j];
  long long inc = loc;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long u = __shfl_up_sync(FULL, inc, o);
    if (lane >= o) inc += u;
  }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  long long woff = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < SCAN_BD / 32; ++w) { const long long x = wsum[w]; woff += (w < warp) ? x : 0; tot += x; }
  long long run = before + woff + inc - loc;
  TO *o = out + row * out_stride;
#pragma unroll
  for (int j = 0; j < SCAN_E; ++j) { if (i0 + j < n) o[i0 + j] = (TO)run; run += v[j]; }
  if (t == ntiles - 1 && tid == 0) {
    // the last tile of the grid may lie beyond a device-side count: its `before` is still the total
    if (total) total[row] = (int32_t)(before + tot);
    if (out_total) o[n] = (TO)(before + tot);
  }
}

static inline int64_t scan_tiles(int64_t n) { return n < 1 ? 1 : (n + SCAN_TILE - 1) / SCAN_TILE; }

// ------------------------------------------------------------------ chain resolution
// tid values while unresolved: >= 0 final id; -1 not a point; <= -2: "same id as column -2-v of
// the row before" (inside a tile) or, once a chunk is done, "same id as column -2-v of the first
// row of this chunk", whose own id is not known yet.
//
// Sequential resolve of `n` rows held in shared memory by ONE warp (lane owns columns lane,
// lane+32, ...): entry <= -2 takes the value of column -2-v of the row before (prev for row 0),
// which is already resolved.  One __syncwarp per row, no block barrier.
__device__ __forceinline__ void warp_resolve_rows(int *rows, int n, int K, const int *prev) {
  const int lane = threadIdx.x & 31;
  for (int i = 0; i < n; ++i) {
    int *r = rows + i * K;
    for (int c = lane; c < K; c += 32) {
      const int v = r[c];
      if (v <= -2) r[c] = prev[-2 - v];
    }
    __syncwarp();
    prev = r;
  }
}

// copy n ints global <-> shared by one warp, 16 bytes per lane and step when both are aligned
__device__ __forceinline__ void warp_copy_ints(int *dst, const int *src, int n) {
  const int lane = threadIdx.x & 31;
  if ((((uintptr_t)dst | (uintptr_t)src) & 15) == 0) {
    const int n4 = n >> 2;
    const int4 *s4 = reinterpret_cast<const int4 *>(src);
    int4 *d4 = reinterpret_cast<int4 *>(dst);
#pragma unroll 4
    for (int e = lane; e < n4; e += 32) d4[e] = s4[e];
    for (int e = (n4 << 2) + lane; e < n; e += 32) dst[e] = src[e];
  } else {
#pragma unroll 4
    for (int e = lane; e < n; e += 32) dst[e] = src[e];
  }
}

__host__ __device__ inline int track_tile_rows(int K) {
  int rt = 4096 / ((K + 31) / 32 * 32);            // <= 16 KB of shared memory per warp
  return rt > 32 ? 32 : (rt < 1 ? 1 : rt);
}

// Sequential pass of ONE warp over rows [r0, r1) of a reference table, tile by tile (<= 32 rows)
// through shared memory: bulk copy in, row after row, bulk copy out.  LINK: the rows come from
// link + base (new partials get their final ids here) and go to T; otherwise T is updated in place.
// A continued entry of row r0 stays a reference (-2 - column) to the row before r0; every later row
// copies what the row before it holds.  `last` (K ints, may be NULL) receives the final row.
template <bool LINK>
__device__ __forceinline__ void warp_chunk_pass(const int32_t *__restrict__ link, const int32_t *__restrict__ base,
                                                int32_t *T, int64_t r0, int64_t r1, int K, int *tile, int RT,
                                                int32_t *last) {
  const int lane = threadIdx.x & 31;
  const int KP = (K + 3) & ~3;                                                  // keeps `rows` 16-byte aligned
  int *rows = tile + KP;                                                        // tile[0..K) = carried row
  for (int64_t t0 = r0; t0 < r1; t0 += RT) {
    const int n = (int)((t0 + RT <= r1) ? RT : r1 - t0);
    warp_copy_ints(rows, (LINK ? link : T) + t0 * K, n * K);
    const int mybase = (LINK && lane < n) ? base[t0 + lane] : 0;
    __syncwarp();
    const int *prev = tile;
    for (int i = 0; i < n; ++i) {
      int *r = rows + i * K;
      const int bi = __shfl_sync(FULL, mybase, i);
      const bool first = (t0 + i == r0);
      for (int c = lane; c < K; c += 32) {
        int v = r[c];
        if (LINK) {
          if (v == LINK_NONE) v = -1;
          else if (v <= -2) v = bi + (-2 - v);         // new partial: final id
          else v = first ? -2 - v : prev[v];           // same id as column v of the row before
        } else if (v <= -2 && !first) {
          v = prev[-2 - v];
        }
        r[c] = v;
      }
      __syncwarp();
      prev = r;
    }
    warp_copy_ints(T + t0 * K, rows, n * K);
    for (int c = lane; c < K; c += 32) tile[c] = rows[(n - 1) * K + c];
    __syncwarp();
  }
  if (last != nullptr) for (int c = lane; c < K; c += 32) last[c] = tile[c];
}

// Chain resolution, hierarchical: every level cuts its table into chunks of RES_CHUNK rows, one warp
// resolves a chunk relative to the row before it (all chunks at once) and hands the chunk's last row
// to the next, RES_CHUNK times shorter level; the last level (<= RES_MID rows) is resolved by one CTA;
// then every level replaces its remaining references by the resolved last row of the chunk before.
constexpr int RES_CHUNK = 32;
constexpr int RES_MID = 512;

__host__ __device__ inline int resolve_tile_ints(int K, int RT) { return (((K + 3) & ~3) + RT * K + 3) & ~3; }

// level 1 (LINK: link + base -> tid) or a higher level (in place); S = last rows of the chunks
template <bool LINK>
__global__ void resolve_chunk_kernel(const int32_t *__restrict__ link, const int32_t *__restrict__ base, int32_t *T,
                                     int64_t n, int K, int RT, int32_t *__restrict__ S) {
  PVK_SMEM(smem);
  const int warp = threadIdx.x >> 5, W = blockDim.x >> 5;
  int *tile = reinterpret_cast<int *>(smem) + (size_t)warp * resolve_tile_ints(K, RT);
  const int64_t ch = (int64_t)blockIdx.x * W + warp;
  const int64_t r0 = ch * RES_CHUNK;
  if (r0 >= n) return;
  const int64_t r1 = r0 + RES_CHUNK < n ? r0 + RES_CHUNK : n;
  warp_chunk_pass<LINK>(link, base, T, r0, r1, K, tile, RT, S + ch * K);
}

// last level: one CTA, warp w owns rows [w m, (w+1) m): chunk pass, then warp 0 walks the NW last rows,
// then every warp resolves what is left in its rows
__global__ void resolve_mid_kernel(int32_t *T, int64_t n, int K, int RT) {
  PVK_SMEM(smem);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, NW = blockDim.x >> 5;
  int *last = reinterpret_cast<int *>(smem);                                    // [NW][K]
  int *tile = last + (((size_t)NW * K + 3) & ~(size_t)3) + (size_t)warp * resolve_tile_ints(K, RT);
  const int64_t m = (n + NW - 1) / NW;
  const int64_t r0 = warp * m, r1 = r0 + m < n ? r0 + m : n;
  if (r0 < n) warp_chunk_pass<false>(nullptr, nullptr, T, r0, r1, K, tile, RT, last + warp * K);
  __syncthreads();
  if (warp == 0) {
    for (int w = 1; w < NW && (int64_t)w * m < n; ++w) {
      for (int c = lane; c < K; c += 32) {
        const int v = last[w * K + c];
        if (v <= -2) last[w * K + c] = last[(w - 1) * K + (-2 - v)];
      }
      __syncwarp();
    }
  }
  __syncthreads();
  if (warp > 0 && r0 < n) {
    const int *pl = last + (warp - 1) * K;
    int32_t *t = T + r0 * K;
    const int64_t ne = (r1 - r0) * K;
    for (int64_t e = lane; e < ne; e += 32) {
      const int v = t[e];
      if (v <= -2) t[e] = pl[-2 - v];
    }
  }
}

// remaining references of chunk i >= 1 -> resolved last row of chunk i - 1 (Sres); one CTA per chunk
__global__ void resolve_fix_kernel(int32_t *__restrict__ T, int64_t n, int K, const int32_t *__restrict__ Sres) {
  for (int64_t ch = 1 + blockIdx.x; ch * RES_CHUNK < n; ch += gridDim.x) {
    const int64_t r0 = ch * RES_CHUNK, r1 = r0 + RES_CHUNK < n ? r0 + RES_CHUNK : n;
    const int32_t *pl = Sres + (ch - 1) * K;
    int32_t *t = T + r0 * K;
    const int ne = (int)((r1 - r0) * K);
    if ((((uintptr_t)t) & 15) == 0 && (ne & 3) == 0) {
      int4 *t4 = reinterpret_cast<int4 *>(t);
      for (int e = threadIdx.x; e < (ne >> 2); e += blockDim.x) {
        int4 v = t4[e];
        if (v.x <= -2 || v.y <= -2 || v.z <= -2 || v.w <= -2) {
          if (v.x <= -2) v.x = pl[-2 - v.x];
          if (v.y <= -2) v.y = pl[-2 - v.y];
          if (v.z <= -2) v.z = pl[-2 - v.z];
          if (v.w <= -2) v.w = pl[-2 - v.w];
          t4[e] = v;
        }
      }
    } else {
      for (int e = threadIdx.x; e < ne; e += blockDim.x) {
        const int v = t[e];
        if (v <= -2) t[e] = pl[-2 - v];
      }
    }
  }
}

// ------------------------------------------------------------------ pack
// Every thread walks one column over a strip of PACK_STRIP consecutive frames and merges runs of
// equal ids (a partial usually stays in its column for a while) before touching the per-track
// counters: ~PACK_STRIP x fewer atomics than one per point.
constexpr int PACK_STRIP = 64;
// Ids >= ntracks (the capacity of tstart / tlen: a speculative pack is sized by an upper bound
// before the real count is known, pv.track_pack_device) are skipped, never written.
__global__ void pack_count_kernel(const int32_t *__restrict__ tid, int64_t F, int K, int64_t ntracks,
                                  int32_t *__restrict__ tstart, int32_t *__restrict__ tlen) {
  const int64_t nstrips = (F + PACK_STRIP - 1) / PACK_STRIP;
  const int64_t n = nstrips * K;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % K);
    const int64_t j0 = (e / K) * PACK_STRIP;
    const int64_t j1 = j0 + PACK_STRIP < F ? j0 + PACK_STRIP : F;
    int cur = -1, cnt = 0;
    int64_t first = 0;
    for (int64_t jb = j0; jb < j1; jb += 8) {                   // 8 independent loads in flight per thread
      int v8[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v8[u] = jb + u < j1 ? tid[(jb + u) * K + c] : -1;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (jb + u < j1) {
          const int v = v8[u];
          if (v != cur) {
            if (cur >= 0 && cur < ntracks) { atomicAdd(&tlen[cur], cnt); atomicMin(&tstart[cur], (int32_t)first); }
            cur = v; cnt = 0; first = jb + u;
          }
          ++cnt;
        }
      }
    }
    if (cur >= 0 && cur < ntracks) { atomicAdd(&tlen[cur], cnt); atomicMin(&tstart[cur], (int32_t)first); }
  }
}

// Tiled scatter: one CTA moves ROWS consecutive frames (one contiguous chunk of every table).  The
// chunk is read coalesced into shared memory and written out with lanes along the FRAME axis: a
// partial keeps its column while the peaks around it are stable, so consecutive frames of one
// column land on consecutive positions of that partial's run -- full-sector stores instead of
// one 8-byte store per 32-byte sector (what a thread-per-element scatter does: 7.7x off the HBM
// bound on the 8 hour configuration, ncu r1k).  Shared memory: int32 pos[ROWS][KP] | double val[ROWS][KP], KP = K | 1.
__global__ void pack_scatter_tiled_kernel(const double *__restrict__ f, const double *__restrict__ mag,
                                          const double *__restrict__ ph, const double *__restrict__ realph,
                                          const int32_t *__restrict__ tid, int64_t F, int K, int ROWS,
                                          int64_t ntracks, int64_t npts_cap,
                                          const int32_t *__restrict__ tstart, const int64_t *__restrict__ toff,
                                          double *__restrict__ pf, double *__restrict__ pmag,
                                          double *__restrict__ pph, double *__restrict__ prealph) {
  PVK_SMEM(smem);
  const int KP = K | 1;
  double *val = reinterpret_cast<double *>(smem);
  int32_t *pos = reinterpret_cast<int32_t *>(smem + (size_t)ROWS * KP * 8);
  const int64_t ntiles = (F + ROWS - 1) / ROWS;
  const int T = blockDim.x, t = threadIdx.x;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t j0 = tile * ROWS;
    const int rows = (int)(F - j0 < ROWS ? F - j0 : ROWS);
    const int64_t base = j0 * K;
    const int n = rows * K;
    for (int e = t; e < n; e += T) {
      const int r = e / K, c = e - r * K;
      const int v = tid[base + e];
      // ids beyond the capacity of the index arrays and positions beyond the packed arrays are dropped
      int64_t q = -1;
      if (v >= 0 && v < ntracks) { q = toff[v] + (j0 + r - tstart[v]); if (q >= npts_cap) q = -1; }
      pos[r * KP + c] = (int32_t)q;
    }
    const double *src[4] = {f, mag, ph, realph};
    double *dst[4] = {pf, pmag, pph, prealph};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (dst[q] == nullptr) continue;                          // uniform
      __syncthreads();                                          // pos ready / previous table written out
      for (int e = t; e < n; e += T) {
        const int r = e / K, c = e - r * K;
        val[r * KP + c] = src[q][base + e];
      }
      __syncthreads();
      for (int e = t; e < ROWS * K; e += T) {                   // lanes along the frame axis
        const int r = e % ROWS, c = e / ROWS;
        if (r < rows) {
          const int p = pos[r * KP + c];
          if (p >= 0) dst[q][p] = val[r * KP + c];
        }
      }
    }
    __syncthreads();
  }
}

// stats[0][clip] = number of points, stats[1][clip] = last frame holding a point (-1: none),
// stats[2][clip] = number of partials: everything the host needs to size the packed tracks and
// the resynthesis, in one read-back
__global__ void track_stats_kernel(const int32_t *__restrict__ tid, const int32_t *__restrict__ ntracks, int64_t F, int K,
                                   long long *__restrict__ stats) {
  const int64_t clip = blockIdx.y, n = F * K;
  const int32_t *t = tid + clip * n;
  long long cnt = 0;
  long long last = -1;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    if (t[e] >= 0) { ++cnt; last = e; }                      // e ascends: the last hit is the largest
  }
  if (last >= 0) last /= K;
  cnt = warp_sum(cnt);
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) { const long long u = __shfl_xor_sync(FULL, last, o); last = u > last ? u : last; }
  if ((threadIdx.x & 31) == 0) {
    if (cnt) atomicAdd(reinterpret_cast<unsigned long long *>(stats + clip), (unsigned long long)cnt);
    if (last >= 0) atomicMax(stats + gridDim.y + clip, last);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) stats[2 * gridDim.y + clip] = ntracks[clip];
}

// Clip batches flattened into one table of rows_per_clip rows per clip (pvk_analyze_batch): per
// clip, the number of partials that start in it and the last LOCAL frame holding a point of one of
// them (-1: none).  Partials never cross a clip (zero guard rows), ids ascend clip after clip.
__global__ void clip_spans_kernel(const int32_t *__restrict__ tstart, const int32_t *__restrict__ tlen, int64_t ntracks,
                                  int64_t rows_per_clip, int64_t nclips, int32_t *__restrict__ count,
                                  int32_t *__restrict__ last) {
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < ntracks; v += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = tstart[v];
    const int64_t c = s / rows_per_clip;
    if (s < 0 || c >= nclips) continue;
    atomicAdd(&count[c], 1);
    atomicMax(&last[c], (int)(s - c * rows_per_clip) + tlen[v] - 1);
  }
}

// ------------------------------------------------------------------ relink (DESIGN.md 4.3, "Remap")
// A table remapped onto output rows by any map tau (pvk_time_map) holds source ids, and a source partial
// read backwards or across a jump covers several runs of consecutive output rows.  The relink gives every
// run its own id, in pvk_track's link encoding, and the scan and resolve of pvk_track number the runs.
//
// col[p] = column of packed point p of the source table: with it, the column of partial v in output row
// b - 1 (= source row floor(tau[b - 1])) is one gather instead of a search of that row.
__global__ void relink_cols_kernel(const int32_t *__restrict__ tid, int64_t n, int K, int64_t ntracks,
                                   const int32_t *__restrict__ tstart, const int32_t *__restrict__ tlen,
                                   const int64_t *__restrict__ toff, int32_t *__restrict__ col) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    const int v = tid[e];
    if (v < 0 || v >= ntracks) continue;
    const int64_t i = e / K;
    const int64_t k = i - tstart[v];
    if (k >= 0 && k < tlen[v]) col[toff[v] + k] = (int32_t)(e - i * K);
  }
}

// One warp per output row b, lanes over columns.  Slot (b, c) holding source partial v continues v's
// run when output row b - 1 holds v, i.e. tstart[v] <= floor(tau[b - 1]) <= end[v]: link = v's column
// there.  Otherwise it starts a run: link = -2 - rank, rank = number of the row's new runs with a smaller
// source id (ids are distinct within a row), so the scan numbers runs by (first output row, source id).
// Shared memory per warp: the row's source ids [K] | one bit per column of a new run [32 words].  Cost per
// row: K coalesced id reads, three gathers and one `col` gather per point, and nnew^2 / 32 shared reads per
// lane for the ranks (nnew = new runs in the row: all points in row 0 and after a jump, few elsewhere).
// The launch bound's 4 CTAs per SM (44 registers) keeps ptxas from holding the kernel at 32 and spilling.
constexpr int RELINK_THREADS = 256;

__host__ __device__ constexpr int relink_smem_per_warp(int K) { return (K + 32) * 4; }

__global__ void __launch_bounds__(RELINK_THREADS, 4) track_relink_kernel(
    const int32_t *__restrict__ tid_map, const double *__restrict__ tmap, int64_t B, int64_t F, int K, int64_t ntracks,
    const int32_t *__restrict__ tstart, const int32_t *__restrict__ tlen, const int64_t *__restrict__ toff,
    const int32_t *__restrict__ col, int32_t *__restrict__ link, int32_t *__restrict__ newcount) {
  PVK_SMEM(smem);
  const int lane = lane_id(), warp = warp_id();
  int *ids = reinterpret_cast<int *>(smem) + (size_t)warp * (K + 32);
  unsigned *bits = reinterpret_cast<unsigned *>(ids + K);
  const int nw = (int)(gridDim.x * (blockDim.x >> 5));              // warps in the grid (<= 148 * 16 * 8)
  for (int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp; b < B; b += nw) {
    const double tp = b > 0 ? tmap[b - 1] : -1.0;
    const int64_t ip = tp >= 0.0 && tp <= (double)(F - 1) ? (int64_t)floor(tp) : -1;   // -1: no row before
    int32_t *lrow = link + b * K;
    int nnew = 0;
    for (int c0 = 0; c0 < K; c0 += 32) {
      const int c = c0 + lane;
      bool fresh = false;
      if (c < K) {
        int v = tid_map[b * K + c];
        int lk = LINK_NONE;
        if (v >= 0 && v < ntracks) {
          const int64_t k = ip - tstart[v];
          if (ip >= 0 && k >= 0 && k < tlen[v]) lk = col[toff[v] + k];
          else fresh = true;
        } else {
          v = -1;
        }
        ids[c] = v;
        if (!fresh) lrow[c] = lk;
      }
      const unsigned m = __ballot_sync(FULL, fresh);
      if (lane == 0) bits[c0 >> 5] = m;
      nnew += __popc(m);
    }
    __syncwarp();
    if (nnew > 0) {
      const int nword = (K + 31) >> 5;
      for (int c = lane; c < K; c += 32) {
        if (!((bits[c >> 5] >> (c & 31)) & 1u)) continue;
        const int v = ids[c];
        int rank = 0;
        for (int w = 0; w < nword; ++w)
          for (unsigned rem = bits[w]; rem; rem &= rem - 1u) rank += ids[32 * w + __ffs((int)rem) - 1] < v ? 1 : 0;
        lrow[c] = -2 - rank;
      }
    }
    if (lane == 0) newcount[b] = nnew;
    __syncwarp();
  }
}

static inline int grid_for(int64_t n, int block) {
  int64_t g = (n + block - 1) / block;
  const int64_t cap = 148 * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace pvk

using namespace pvk;

// last-row tables of all resolve levels: rows/32 + rows/32^2 + ... rows of npks ints
static int64_t resolve_levels_bytes(int64_t rows, int npks) {
  int64_t total = 0;
  for (int64_t n = rows; n > 1;) {
    n = (n + RES_CHUNK - 1) / RES_CHUNK;
    total += align_up(n * npks * 4, 256);
  }
  return total + 256;
}

extern "C" int64_t pvk_track_workspace_bytes(int64_t nclips, int64_t nframes, int npks) {
  if (nclips < 0 || nframes < 0 || npks < 1) return -1;
  const int64_t rows = nclips * nframes;
  return align_up(rows * 4, 256) * 2 + resolve_levels_bytes(rows, npks) +
         align_up(nclips * scan_tiles(nframes) * 8, 256) + 256;
}

// The numbering half of pvk_track, shared with pvk_track_relink: the per-clip exclusive scan of the
// rows' new-partial counts (newcount -> base, ntracks), then the chain resolution that turns link + base
// into ids (tid).  `name` is the export's name for error messages.
#define PVK_CHECK_STAGE(stage)                                                                      \
  do {                                                                                              \
    char _what[64];                                                                                 \
    snprintf(_what, sizeof _what, "%s(" stage ")", name);                                          \
    PVK_CHECK_LAUNCH(_what);                                                                        \
  } while (0)

static int track_number(const int32_t *link, int32_t *newcount, int32_t *base, unsigned char *levels, long long *tsum,
                        int64_t nclips, int64_t nframes, int K, int32_t *tid, int32_t *ntracks, void *stream,
                        const char *name) {
  const int64_t rows = nclips * nframes;
  {
    const int64_t nt = scan_tiles(nframes);
    PVK_REQUIRE(nclips <= 65535, "%s: at most 65535 clips per call (got %lld)", name, (long long)nclips);
    PVK_LAUNCH(scan_tile_sums_kernel, dim3((unsigned)nt, (unsigned)nclips), dim3(SCAN_BD), SCAN_SMEM, stream, newcount, nframes,
               nframes, (const int32_t *)nullptr, nt, tsum);
    PVK_LAUNCH(scan_tile_apply_kernel<int32_t>, dim3((unsigned)nt, (unsigned)nclips), dim3(SCAN_BD), SCAN_SMEM, stream, newcount,
               nframes, nframes, (const int32_t *)nullptr, nt, tsum, base, nframes, ntracks, 0);
    PVK_CHECK_STAGE("scan");
  }
  {
    // ---- chain resolution: level 1 turns link + base into ids chunk by chunk, the chunks' last rows
    //      form the next level, ... the last level is resolved by one CTA, then the references left in
    //      every level are replaced top-down.  The first row of every clip holds no reference.
    const int RT = track_tile_rows(K);
    const size_t per_warp = (size_t)resolve_tile_ints(K, RT) * 4;
    int W = (int)((64 * 1024) / per_warp);
    if (W > 4) W = 4;
    if (W < 1) W = 1;
    const size_t csm = per_warp * W;
    if (csm > 48 * 1024 && (PVK_SET_SMEM(resolve_chunk_kernel<true>, (int)csm) != 0 ||
                            PVK_SET_SMEM(resolve_chunk_kernel<false>, (int)csm) != 0)) {
      set_error("%s: cannot reserve %d bytes of shared memory", name, (int)csm);
      return PVK_ERR_CUDA;
    }
    int32_t *tab[16];
    int64_t len[16];
    int nl = 0;
    tab[0] = tid; len[0] = rows;
    unsigned char *lp = levels;
    {
      const int64_t nch = (rows + RES_CHUNK - 1) / RES_CHUNK;
      tab[1] = reinterpret_cast<int32_t *>(lp); len[1] = nch;
      lp += align_up(nch * K * 4, 256);
      PVK_LAUNCH(resolve_chunk_kernel<true>, dim3((unsigned)((nch + W - 1) / W)), dim3(W * 32), csm, stream, link, base,
                 tid, rows, K, RT, tab[1]);
      PVK_CHECK_STAGE("chunk");
      nl = 1;
    }
    if (len[1] > 1) {
      while (len[nl] > RES_MID) {
        const int64_t nch = (len[nl] + RES_CHUNK - 1) / RES_CHUNK;
        tab[nl + 1] = reinterpret_cast<int32_t *>(lp); len[nl + 1] = nch;
        lp += align_up(nch * K * 4, 256);
        PVK_LAUNCH(resolve_chunk_kernel<false>, dim3((unsigned)((nch + W - 1) / W)), dim3(W * 32), csm, stream,
                   (const int32_t *)nullptr, (const int32_t *)nullptr, tab[nl], len[nl], K, RT, tab[nl + 1]);
        PVK_CHECK_STAGE("chunk");
        ++nl;
      }
      {
        int NW = K > 512 ? 8 : 16;
        int RTm = RT;
        while (RTm > 1 && ((size_t)NW * K + 4 + (size_t)NW * resolve_tile_ints(K, RTm)) * 4 > 160 * 1024) RTm >>= 1;
        const size_t msm = ((((size_t)NW * K + 3) & ~(size_t)3) + (size_t)NW * resolve_tile_ints(K, RTm)) * 4;
        if (msm > 48 * 1024 && PVK_SET_SMEM(resolve_mid_kernel, (int)msm) != 0) {
          set_error("%s: cannot reserve %d bytes of shared memory", name, (int)msm);
          return PVK_ERR_CUDA;
        }
        PVK_LAUNCH(resolve_mid_kernel, dim3(1), dim3(NW * 32), msm, stream, tab[nl], len[nl], K, RTm);
        PVK_CHECK_STAGE("mid");
      }
      for (int l = nl - 1; l >= 0; --l) {
        int64_t g = (len[l] + RES_CHUNK - 1) / RES_CHUNK - 1;
        if (g < 1) continue;
        if (g > 148 * 32) g = 148 * 32;
        PVK_LAUNCH(resolve_fix_kernel, dim3((unsigned)g), dim3(128), 0, stream, tab[l], len[l], K, tab[l + 1]);
        PVK_CHECK_STAGE("fix");
      }
    }
  }
  return PVK_OK;
}
#undef PVK_CHECK_STAGE

extern "C" int pvk_track(const double *f, const double *mag, int64_t nclips, int64_t nframes, int npks,
                         double maxpitchjmp, int32_t *tid, int32_t *link, int32_t *ntracks,
                         void *workspace, int64_t workspace_bytes, void *stream) {
  PVK_REQUIRE(npks >= 1 && npks <= PVK_MAX_NPKS, "pvk_track: npks=%d must be in [1, %d]", npks, PVK_MAX_NPKS);
  PVK_REQUIRE(nclips >= 0 && nframes >= 0, "pvk_track: negative sizes");
  PVK_REQUIRE(ntracks != nullptr, "pvk_track: ntracks is NULL");
  if (nclips == 0) return PVK_OK;
  if (nframes == 0) {
    cudaMemsetAsync(ntracks, 0, (size_t)nclips * 4, (cudaStream_t)stream);
    return PVK_OK;
  }
  PVK_REQUIRE(f && mag && tid && link && workspace, "pvk_track: NULL pointer argument");
  PVK_REQUIRE(workspace_bytes >= pvk_track_workspace_bytes(nclips, nframes, npks),
              "pvk_track: workspace too small (%lld < %lld bytes)", (long long)workspace_bytes,
              (long long)pvk_track_workspace_bytes(nclips, nframes, npks));
  PVK_REQUIRE(nclips * nframes * (int64_t)npks < (int64_t)2147483647,
              "pvk_track: nclips*nframes*npks must be < 2^31");
  const int K = npks;
  const int64_t rows = nclips * nframes;
  unsigned char *ws = reinterpret_cast<unsigned char *>(workspace);
  int32_t *newcount = reinterpret_cast<int32_t *>(ws);
  int32_t *base = reinterpret_cast<int32_t *>(ws + align_up(rows * 4, 256));
  unsigned char *levels = ws + 2 * align_up(rows * 4, 256);
  long long *tsum = reinterpret_cast<long long *>(levels + resolve_levels_bytes(rows, npks));

  {  // link: one warp per frame pair
    int64_t g;
    // up to 128 peaks: one warp per row; up to 512: one CTA per row; wider rows: the sequential loop kernel
    if (K <= 128) {
      const int S = K <= 32 ? 1 : (K <= 64 ? 2 : 4);
      const int W = 8;
      const int smem = W * link_claim_smem_per_warp(S);
      g = (rows + W - 1) / W;
      if (g > 148 * 64) g = 148 * 64;
#define PVK_LINK_CLAIM(SS)                                                                         \
      do {                                                                                           \
        if (smem > 48 * 1024 && PVK_SET_SMEM(track_link_claim_kernel<SS>, smem) != 0) {             \
          set_error("pvk_track: cannot reserve %d bytes of shared memory", smem);                    \
          return PVK_ERR_CUDA;                                                                       \
        }                                                                                            \
        PVK_LAUNCH(track_link_claim_kernel<SS>, dim3((unsigned)g), dim3(W * 32), smem, stream, f, mag, rows, \
                   nframes, K, maxpitchjmp, link, newcount);                                         \
      } while (0)
      if (S == 1) PVK_LINK_CLAIM(1);
      else if (S == 2) PVK_LINK_CLAIM(2);
      else PVK_LINK_CLAIM(4);
#undef PVK_LINK_CLAIM
    } else if (K <= 512) {
      // one CTA per row: 128 threads up to 256 columns, 256 threads up to 512
      const int T = K <= 256 ? 128 : 256;
      const int smem = link_cta_smem(2 * T);
      if (smem > 48 * 1024 && PVK_SET_SMEM(track_link_cta_kernel, smem) != 0) {
        set_error("pvk_track: cannot reserve %d bytes of shared memory", smem);
        return PVK_ERR_CUDA;
      }
      g = rows < 148 * 16 ? rows : 148 * 16;
      PVK_LAUNCH(track_link_cta_kernel, dim3((unsigned)g), dim3(T), smem, stream, f, mag, rows, nframes, K, maxpitchjmp,
                 link, newcount);
    } else {
      const int per_warp = link_generic_smem_per_warp(K);
      int W = 96 * 1024 / per_warp;                               // two CTAs per SM
      if (W > 8) W = 8;
      if (W < 1) W = 1;
      const int smem = W * per_warp;
      if (smem > 48 * 1024) {
        if (PVK_SET_SMEM(track_link_kernel, smem) != 0) {
          set_error("pvk_track: cannot reserve %d bytes of shared memory", smem);
          return PVK_ERR_CUDA;
        }
      }
      g = (rows + W - 1) / W;
      if (g > 148 * 64) g = 148 * 64;
      PVK_LAUNCH(track_link_kernel, dim3((unsigned)g), dim3(W * 32), smem, stream, f, mag, rows, nframes, K,
                 maxpitchjmp, link, newcount);
    }
    PVK_CHECK_LAUNCH("pvk_track(link)");
  }
  return track_number(link, newcount, base, levels, tsum, nclips, nframes, K, tid, ntracks, stream, "pvk_track");
}

// pvk_track's workspace for one clip of nrows_out rows, then the source column of every packed point
extern "C" int64_t pvk_track_relink_workspace_bytes(int64_t nframes, int npks, int64_t nrows_out) {
  if (nframes < 0 || npks < 1 || nrows_out < 0) return -1;
  return pvk_track_workspace_bytes(1, nrows_out, npks) + align_up(nframes * npks * 4, 256);
}

extern "C" int pvk_track_relink(const int32_t *tid_src, int64_t nframes, int npks, int64_t ntracks_src,
                                const int32_t *tstart, const int32_t *tlen, const int64_t *toff, const int32_t *tid_map,
                                const double *tmap, int64_t nrows_out, int32_t *tid_out, int32_t *link_out,
                                int32_t *ntracks_out, void *workspace, int64_t workspace_bytes, void *stream) {
  PVK_REQUIRE(npks >= 1 && npks <= PVK_MAX_NPKS, "pvk_track_relink: npks=%d must be in [1, %d]", npks, PVK_MAX_NPKS);
  PVK_REQUIRE(nframes >= 0 && ntracks_src >= 0 && nrows_out >= 0, "pvk_track_relink: negative sizes");
  PVK_REQUIRE(ntracks_out != nullptr, "pvk_track_relink: ntracks_out is NULL");
  PVK_REQUIRE(nrows_out * (int64_t)npks < (int64_t)2147483647 && nframes * (int64_t)npks < (int64_t)2147483647,
              "pvk_track_relink: nrows_out*npks and nframes*npks must be < 2^31");
  if (nrows_out == 0) {
    cudaMemsetAsync(ntracks_out, 0, 4, (cudaStream_t)stream);
    return PVK_OK;
  }
  PVK_REQUIRE(nframes >= 1, "pvk_track_relink: a remap needs a source table with at least one frame row");
  PVK_REQUIRE(tid_src && tid_map && tmap && tid_out && link_out && workspace &&
                  (ntracks_src == 0 || (tstart && tlen && toff)),
              "pvk_track_relink: NULL pointer argument");
  const int64_t need = pvk_track_relink_workspace_bytes(nframes, npks, nrows_out);
  PVK_REQUIRE(workspace_bytes >= need, "pvk_track_relink: workspace too small (%lld < %lld bytes)",
              (long long)workspace_bytes, (long long)need);
  const int K = npks;
  const int64_t B = nrows_out;
  unsigned char *ws = reinterpret_cast<unsigned char *>(workspace);
  int32_t *newcount = reinterpret_cast<int32_t *>(ws);
  int32_t *base = reinterpret_cast<int32_t *>(ws + align_up(B * 4, 256));
  unsigned char *levels = ws + 2 * align_up(B * 4, 256);
  long long *tsum = reinterpret_cast<long long *>(levels + resolve_levels_bytes(B, npks));
  int32_t *col = reinterpret_cast<int32_t *>(ws + pvk_track_workspace_bytes(1, B, npks));
  if (ntracks_src > 0) {
    PVK_LAUNCH(relink_cols_kernel, dim3(grid_for(nframes * K, 256)), dim3(256), 0, stream, tid_src, nframes * K, K,
               ntracks_src, tstart, tlen, toff, col);
    PVK_CHECK_LAUNCH("pvk_track_relink(cols)");
  }
  {
    const int W = RELINK_THREADS / 32;
    const int smem = W * relink_smem_per_warp(K);
    const int64_t g = (B + W - 1) / W < 148 * 16 ? (B + W - 1) / W : 148 * 16;
    PVK_LAUNCH(track_relink_kernel, dim3((unsigned)g), dim3(RELINK_THREADS), smem, stream, tid_map, tmap, B, nframes, K,
               ntracks_src, tstart, tlen, toff, col, link_out, newcount);
    PVK_CHECK_LAUNCH("pvk_track_relink(link)");
  }
  return track_number(link_out, newcount, base, levels, tsum, 1, B, K, tid_out, ntracks_out, stream,
                      "pvk_track_relink");
}

extern "C" int pvk_track_spans(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks, int32_t *tstart,
                               int32_t *tlen, void *stream) {
  PVK_REQUIRE(npks >= 1 && nframes >= 0 && ntracks >= 0, "pvk_track_spans: bad sizes");
  if (ntracks == 0) return PVK_OK;
  PVK_REQUIRE(tstart && tlen, "pvk_track_spans: NULL pointer argument");
  cudaMemsetAsync(tlen, 0, 4 * (size_t)ntracks, (cudaStream_t)stream);
  cudaMemsetAsync(tstart, 0x7f, 4 * (size_t)ntracks, (cudaStream_t)stream);   // 0x7f7f7f7f: "no frame yet"
  if (nframes == 0) return PVK_OK;
  PVK_REQUIRE(tid != nullptr, "pvk_track_spans: tid is NULL");
  PVK_LAUNCH(pack_count_kernel, dim3(grid_for((nframes + PACK_STRIP - 1) / PACK_STRIP * npks, 128)), dim3(128), 0,
             stream, tid, nframes, npks, ntracks, tstart, tlen);
  PVK_CHECK_LAUNCH("pvk_track_spans");
  return PVK_OK;
}

extern "C" int pvk_track_stats(const int32_t *tid, const int32_t *ntracks, int64_t nclips, int64_t nframes, int npks,
                               int64_t *stats, void *stream) {
  PVK_REQUIRE(npks >= 1 && nframes >= 0 && nclips >= 0 && nclips <= 65535, "pvk_track_stats: bad sizes");
  if (nclips == 0) return PVK_OK;
  PVK_REQUIRE(stats && ntracks && (tid || nframes == 0), "pvk_track_stats: NULL pointer argument");
  cudaMemsetAsync(stats, 0, (size_t)nclips * 8, (cudaStream_t)stream);
  cudaMemsetAsync(stats + nclips, 0xff, (size_t)nclips * 8, (cudaStream_t)stream);        // -1
  int g = grid_for(nframes * npks, 256);
  if (g > 148 * 4) g = 148 * 4;
  PVK_LAUNCH(track_stats_kernel, dim3((unsigned)g, (unsigned)nclips), dim3(256), 0, stream, tid, ntracks, nframes, npks,
             reinterpret_cast<long long *>(stats));
  PVK_CHECK_LAUNCH("pvk_track_stats");
  return PVK_OK;
}

extern "C" int pvk_clip_spans(const int32_t *tstart, const int32_t *tlen, int64_t ntracks, int64_t rows_per_clip,
                              int64_t nclips, int32_t *count, int32_t *last, void *stream) {
  PVK_REQUIRE(ntracks >= 0 && rows_per_clip >= 1 && nclips >= 0, "pvk_clip_spans: bad sizes");
  if (nclips == 0) return PVK_OK;
  PVK_REQUIRE(count && last && (ntracks == 0 || (tstart && tlen)), "pvk_clip_spans: NULL pointer argument");
  cudaMemsetAsync(count, 0, 4 * (size_t)nclips, (cudaStream_t)stream);
  cudaMemsetAsync(last, 0xff, 4 * (size_t)nclips, (cudaStream_t)stream);                 // -1
  if (ntracks == 0) return PVK_OK;
  PVK_LAUNCH(clip_spans_kernel, dim3(grid_for(ntracks, 256)), dim3(256), 0, stream, tstart, tlen, ntracks, rows_per_clip,
             nclips, count, last);
  PVK_CHECK_LAUNCH("pvk_clip_spans");
  return PVK_OK;
}

extern "C" int64_t pvk_track_pack_workspace_bytes(int64_t ntracks) {
  if (ntracks < 0) return -1;
  return align_up(scan_tiles(ntracks) * 8, 256);
}

extern "C" int pvk_track_pack(const double *f, const double *mag, const double *ph, const double *realph,
                              const int32_t *tid, int64_t nframes, int npks,
                              int64_t ntracks, int32_t *tstart, int32_t *tlen, int64_t *toff, double *pf,
                              double *pmag, double *pph, double *prealph, void *workspace,
                              int64_t workspace_bytes, void *stream) {
  return pvk_track_pack_dev(f, mag, ph, realph, tid, nframes, npks, ntracks, nullptr, tstart, tlen, toff, pf, pmag, pph,
                            prealph, workspace, workspace_bytes, stream);
}

extern "C" int pvk_track_pack_dev(const double *f, const double *mag, const double *ph, const double *realph,
                                  const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                                  const int32_t *ntracks_dev, int32_t *tstart, int32_t *tlen, int64_t *toff,
                                  double *pf, double *pmag, double *pph, double *prealph, void *workspace,
                                  int64_t workspace_bytes, void *stream) {
  PVK_REQUIRE(npks >= 1 && nframes >= 0 && ntracks >= 0, "pvk_track_pack: bad sizes");
  PVK_REQUIRE(toff != nullptr, "pvk_track_pack: toff is NULL");
  if (ntracks == 0 || nframes == 0) {
    cudaMemsetAsync(toff, 0, 8 * (size_t)(ntracks + 1), (cudaStream_t)stream);
    return PVK_OK;
  }
  PVK_REQUIRE(f && mag && realph && tid && tstart && tlen && pf && pmag && prealph,
              "pvk_track_pack: NULL pointer argument");
  PVK_REQUIRE(workspace != nullptr && workspace_bytes >= pvk_track_pack_workspace_bytes(ntracks),
              "pvk_track_pack: workspace too small (%lld bytes; pvk_track_pack_workspace_bytes gives the size)",
              (long long)workspace_bytes);
  const int64_t n = nframes * npks;
  cudaMemsetAsync(tlen, 0, 4 * (size_t)ntracks, (cudaStream_t)stream);
  cudaMemsetAsync(tstart, 0x7f, 4 * (size_t)ntracks, (cudaStream_t)stream);   // 0x7f7f7f7f: "no frame yet"
  PVK_LAUNCH(pack_count_kernel, dim3(grid_for((nframes + PACK_STRIP - 1) / PACK_STRIP * npks, 128)), dim3(128), 0,
             stream, tid, nframes, npks, ntracks, tstart, tlen);
  PVK_CHECK_LAUNCH("pvk_track_pack(count)");
  {
    const int64_t nt = scan_tiles(ntracks);
    long long *tsum = reinterpret_cast<long long *>(workspace);
    PVK_LAUNCH(scan_tile_sums_kernel, dim3((unsigned)nt), dim3(SCAN_BD), SCAN_SMEM, stream, tlen, ntracks, ntracks,
               ntracks_dev, nt, tsum);
    PVK_LAUNCH(scan_tile_apply_kernel<int64_t>, dim3((unsigned)nt), dim3(SCAN_BD), SCAN_SMEM, stream, tlen, ntracks, ntracks,
               ntracks_dev, nt, tsum, toff, ntracks + 1, (int32_t *)nullptr, 1);
    PVK_CHECK_LAUNCH("pvk_track_pack(scan)");
  }
  {
    // rows per tile: as many as fit ~96 KB of shared memory (12 bytes per padded slot), at most 32
    const int KP = npks | 1;
    int rows = 32;
    while (rows > 1 && (size_t)rows * KP * 12 > 96 * 1024) rows >>= 1;
    const int smem = rows * KP * 12;
    const int64_t ntiles = (nframes + rows - 1) / rows;
    if (smem > 48 * 1024 && PVK_SET_SMEM(pack_scatter_tiled_kernel, smem) != 0) {
      set_error("pvk_track_pack: cannot reserve %d bytes of shared memory", smem);
      return PVK_ERR_CUDA;
    }
    int64_t g = ntiles < 148 * 16 ? ntiles : 148 * 16;
    PVK_LAUNCH(pack_scatter_tiled_kernel, dim3((unsigned)g), dim3(256), smem, stream, f, mag, ph, realph, tid, nframes,
               npks, rows, ntracks, n, tstart, toff, pf, pmag, pph, prealph);
  }
  (void)n;
  PVK_CHECK_LAUNCH("pvk_track_pack(scatter)");
  return PVK_OK;
}

// ------------------------------------------------------------------ segment sharding helpers
// (pypevoc_b200/dist.py: global numbering of partials that were linked per segment)
namespace pvk {

// summary[0..K) local ids of the row before the first own row, [K..2K) of the last own row,
// [2K] nb = partials born before the own rows, [2K+1] nb + n_own, [2K+2] global index of the last
// own row holding a point, [2K+3] number of own rows.  Pre-set to -1 / 0 by the caller.
// summary <- {-1 x 2K, 0, 0, -1, nown}: set on the device (no pageable host-to-device copy: nothing that
// could synchronise the side stream the call sits on, and capturable in a CUDA graph)
__global__ void segment_summary_init_kernel(int32_t *__restrict__ summary, int K, int32_t nown) {
  for (int c = threadIdx.x; c < 2 * K + 4; c += blockDim.x)
    summary[c] = c < 2 * K ? -1 : (c == 2 * K + 2 ? -1 : (c == 2 * K + 3 ? nown : 0));
}

__global__ void segment_summary_kernel(const int32_t *__restrict__ tid, int K, int64_t own0, int64_t nown,
                                       int64_t j0, int32_t *__restrict__ summary) {
  const int64_t n = (own0 + nown) * K;
  int mb = -1, mo = -1, lastrow = -1;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    const int v = tid[e];
    const int64_t row = e / K;
    if (row < own0) mb = max(mb, v);
    else if (v >= 0) { mo = max(mo, v); lastrow = max(lastrow, (int)(row - own0)); }
    if (row == own0 - 1) summary[e - row * K] = v;
    if (row == own0 + nown - 1) summary[K + (e - row * K)] = v;
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    mb = max(mb, __shfl_xor_sync(FULL, mb, o));
    mo = max(mo, __shfl_xor_sync(FULL, mo, o));
    lastrow = max(lastrow, __shfl_xor_sync(FULL, lastrow, o));
  }
  if ((threadIdx.x & 31) == 0) {
    if (mb >= 0) { atomicMax(&summary[2 * K], mb + 1); atomicMax(&summary[2 * K + 1], mb + 1); }
    if (mo >= 0) atomicMax(&summary[2 * K + 1], mo + 1);
    if (lastrow >= 0) atomicMax(&summary[2 * K + 2], (int)(j0 + lastrow));
  }
}

// Sequential pass over the ranks (one CTA): global ids of the row before `rank`'s first own row,
// expressed per local id (gidlow[v] for the local ids v < nb born in the back halo), and
// params = {base, nb, n_own, total partials, global index of the last frame with a point}.
__global__ void segment_resolve_kernel(const int32_t *__restrict__ summ, int world, int K, int rank,
                                       int32_t *__restrict__ inv, int cap, int32_t *__restrict__ gidlow,
                                       int32_t *__restrict__ params) {
  PVK_SMEM(smem);
  int *G = reinterpret_cast<int *>(smem);          // [K] global ids of the previous rank's last own row
  int *Gn = G + K;
  const int t = threadIdx.x, BD = blockDim.x;
  for (int c = t; c < K; c += BD) G[c] = -1;
  int base = 0, maxend = -1;
  __syncthreads();
  for (int g = 0; g < world; ++g) {
    const int32_t *s = summ + (int64_t)g * (2 * K + 4);
    const int nb = s[2 * K], nbo = s[2 * K + 1], lastrow = s[2 * K + 2], nown = s[2 * K + 3];
    if (nown == 0) continue;                        // uniform
    const int n_own = nbo - nb;
    for (int c = t; c < K; c += BD) { const int pt = s[c]; if (pt >= 0 && pt < cap) inv[pt] = c; }
    __syncthreads();
    if (g == rank) {
      for (int c = t; c < K; c += BD) { const int pt = s[c]; if (pt >= 0 && pt < cap) gidlow[pt] = G[c]; }
      if (t == 0) { params[0] = base; params[1] = nb; params[2] = n_own; }
    }
    for (int c = t; c < K; c += BD) {
      const int lt = s[K + c];
      Gn[c] = lt < 0 ? -1 : (lt >= nb ? base + (lt - nb) : (lt < cap ? G[inv[lt]] : -1));
    }
    __syncthreads();
    for (int c = t; c < K; c += BD) G[c] = Gn[c];
    base += n_own;
    maxend = max(maxend, lastrow);
    __syncthreads();
  }
  if (t == 0) { params[3] = base; params[4] = maxend; }
}

__global__ void segment_rename_kernel(const int32_t *__restrict__ tid_own, int64_t n, const int32_t *__restrict__ gidlow,
                                      const int32_t *__restrict__ params, int32_t *__restrict__ out) {
  const int base = params[0], nb = params[1];
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    const int v = tid_own[e];
    out[e] = v < 0 ? -1 : (v >= nb ? base + (v - nb) : gidlow[v]);
  }
}

// segment_rename fused with the gather of the track table: every renamed id is stored into the
// table of EVERY rank at the segment's row offset.  dst[d] are int32 tables of all ranks -- the local
// one and peer memory mapped over NVLink (CUDA IPC / symmetric memory) -- so the exchange is plain
// P2P stores issued by the kernel that computes the ids, 128 bits at a time where alignment allows;
// no collective call.  The caller brackets the launch with its cross-rank barriers.
__global__ void segment_rename_push_kernel(const int32_t *__restrict__ tid_own, int64_t n,
                                           const int32_t *__restrict__ gidlow, const int32_t *__restrict__ params,
                                           int32_t *const *__restrict__ dst, int ndst, int64_t offset) {
  const int base = params[0], nb = params[1];
  const bool vec = (offset & 3) == 0 && (reinterpret_cast<uintptr_t>(tid_own) & 15) == 0;
  const int64_t n4 = vec ? n >> 2 : 0;
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, ts = (int64_t)gridDim.x * blockDim.x;
  for (int64_t q = t0; q < n4; q += ts) {
    const int4 v = reinterpret_cast<const int4 *>(tid_own)[q];
    int4 o;
    o.x = v.x < 0 ? -1 : (v.x >= nb ? base + (v.x - nb) : gidlow[v.x]);
    o.y = v.y < 0 ? -1 : (v.y >= nb ? base + (v.y - nb) : gidlow[v.y]);
    o.z = v.z < 0 ? -1 : (v.z >= nb ? base + (v.z - nb) : gidlow[v.z]);
    o.w = v.w < 0 ? -1 : (v.w >= nb ? base + (v.w - nb) : gidlow[v.w]);
    for (int d = 0; d < ndst; ++d) {
      int32_t *t = dst[d] + offset;
      if ((reinterpret_cast<uintptr_t>(t) & 15) == 0) reinterpret_cast<int4 *>(t)[q] = o;
      else { t[4 * q] = o.x; t[4 * q + 1] = o.y; t[4 * q + 2] = o.z; t[4 * q + 3] = o.w; }
    }
  }
  for (int64_t e = 4 * n4 + t0; e < n; e += ts) {
    const int v = tid_own[e];
    const int o = v < 0 ? -1 : (v >= nb ? base + (v - nb) : gidlow[v]);
    for (int d = 0; d < ndst; ++d) dst[d][offset + e] = o;
  }
}

// The same through NVSwitch MULTICAST: `mc` is the multicast address of the ranks' tables (one
// symmetric allocation bound to a multicast object); one multimem.st leaves the GPU once and the
// switch replicates it into the table of every rank, this one included -- 1/N of the NVLink egress
// of per-peer stores.
__device__ __forceinline__ void mc_store4(int32_t *p, int4 o) {
#ifdef PVK_EMU
  *reinterpret_cast<int4 *>(p) = o;
#else
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(__int_as_float(o.x)),
               "f"(__int_as_float(o.y)), "f"(__int_as_float(o.z)), "f"(__int_as_float(o.w))
               : "memory");
#endif
}
__device__ __forceinline__ void mc_store1(int32_t *p, int o) {
#ifdef PVK_EMU
  *p = o;
#else
  asm volatile("multimem.st.relaxed.sys.global.f32 [%0], %1;" ::"l"(p), "f"(__int_as_float(o)) : "memory");
#endif
}

__global__ void segment_rename_mcast_kernel(const int32_t *__restrict__ tid_own, int64_t n,
                                            const int32_t *__restrict__ gidlow, const int32_t *__restrict__ params,
                                            int32_t *mc, int64_t offset) {
  const int base = params[0], nb = params[1];
  int32_t *t = mc + offset;
  const bool vec = (reinterpret_cast<uintptr_t>(t) & 15) == 0 && (reinterpret_cast<uintptr_t>(tid_own) & 15) == 0;
  const int64_t n4 = vec ? n >> 2 : 0;
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, ts = (int64_t)gridDim.x * blockDim.x;
  for (int64_t q = t0; q < n4; q += ts) {
    const int4 v = reinterpret_cast<const int4 *>(tid_own)[q];
    int4 o;
    o.x = v.x < 0 ? -1 : (v.x >= nb ? base + (v.x - nb) : gidlow[v.x]);
    o.y = v.y < 0 ? -1 : (v.y >= nb ? base + (v.y - nb) : gidlow[v.y]);
    o.z = v.z < 0 ? -1 : (v.z >= nb ? base + (v.z - nb) : gidlow[v.z]);
    o.w = v.w < 0 ? -1 : (v.w >= nb ? base + (v.w - nb) : gidlow[v.w]);
    mc_store4(t + 4 * q, o);
  }
  for (int64_t e = 4 * n4 + t0; e < n; e += ts) {
    const int v = tid_own[e];
    mc_store1(t + e, v < 0 ? -1 : (v >= nb ? base + (v - nb) : gidlow[v]));
  }
}

}  // namespace pvk

extern "C" int pvk_segment_summary(const int32_t *tid, int npks, int64_t own0, int64_t nown, int64_t j0,
                                   int32_t *summary, void *stream) {
  PVK_REQUIRE(npks >= 1 && own0 >= 0 && nown >= 0 && summary, "pvk_segment_summary: bad arguments");
  const int K = npks;
  PVK_LAUNCH(segment_summary_init_kernel, dim3(1), dim3(256), 0, stream, summary, K, (int32_t)nown);
  PVK_CHECK_LAUNCH("pvk_segment_summary");
  if (nown == 0) return PVK_OK;
  PVK_REQUIRE(tid != nullptr, "pvk_segment_summary: tid is NULL");
  PVK_LAUNCH(segment_summary_kernel, dim3(grid_for((own0 + nown) * K, 256)), dim3(256), 0, stream, tid, K, own0, nown,
             j0, summary);
  PVK_CHECK_LAUNCH("pvk_segment_summary");
  return PVK_OK;
}

extern "C" int pvk_segment_resolve(const int32_t *summaries, int world, int npks, int rank, int32_t *scratch,
                                   int64_t scratch_ints, int32_t *gidlow, int32_t *params, void *stream) {
  PVK_REQUIRE(summaries && scratch && gidlow && params && world >= 1 && rank >= 0 && rank < world && npks >= 1,
              "pvk_segment_resolve: bad arguments");
  PVK_REQUIRE(scratch_ints >= 1 && scratch_ints < (int64_t)2147483647, "pvk_segment_resolve: bad scratch size");
  const int bd = npks < 1024 ? (npks + 31) / 32 * 32 : 1024;
  PVK_LAUNCH(segment_resolve_kernel, dim3(1), dim3(bd), (size_t)npks * 8, stream, summaries, world, npks, rank, scratch,
             (int)scratch_ints, gidlow, params);
  PVK_CHECK_LAUNCH("pvk_segment_resolve");
  return PVK_OK;
}

extern "C" int pvk_segment_rename(const int32_t *tid_own, int64_t n, const int32_t *gidlow, const int32_t *params,
                                  int32_t *tid_global, void *stream) {
  PVK_REQUIRE(n >= 0, "pvk_segment_rename: negative size");
  if (n == 0) return PVK_OK;
  PVK_REQUIRE(tid_own && gidlow && params && tid_global, "pvk_segment_rename: NULL pointer argument");
  PVK_LAUNCH(segment_rename_kernel, dim3(grid_for(n, 256)), dim3(256), 0, stream, tid_own, n, gidlow, params, tid_global);
  PVK_CHECK_LAUNCH("pvk_segment_rename");
  return PVK_OK;
}

extern "C" int pvk_segment_rename_push(const int32_t *tid_own, int64_t n, const int32_t *gidlow, const int32_t *params,
                                       int32_t *const *dst_tables, int ndst, int64_t dst_offset, void *stream) {
  PVK_REQUIRE(n >= 0 && ndst >= 1 && dst_offset >= 0, "pvk_segment_rename_push: bad sizes");
  if (n == 0) return PVK_OK;
  PVK_REQUIRE(tid_own && gidlow && params && dst_tables, "pvk_segment_rename_push: NULL pointer argument");
  PVK_LAUNCH(segment_rename_push_kernel, dim3(grid_for(n / 4 + 1, 256)), dim3(256), 0, stream, tid_own, n, gidlow, params,
             dst_tables, ndst, dst_offset);
  PVK_CHECK_LAUNCH("pvk_segment_rename_push");
  return PVK_OK;
}

extern "C" int pvk_segment_rename_mcast(const int32_t *tid_own, int64_t n, const int32_t *gidlow, const int32_t *params,
                                        int32_t *mc_table, int64_t dst_offset, void *stream) {
  PVK_REQUIRE(n >= 0 && dst_offset >= 0, "pvk_segment_rename_mcast: bad sizes");
  if (n == 0) return PVK_OK;
  PVK_REQUIRE(tid_own && gidlow && params && mc_table, "pvk_segment_rename_mcast: NULL pointer argument");
  PVK_LAUNCH(segment_rename_mcast_kernel, dim3(grid_for(n / 4 + 1, 256)), dim3(256), 0, stream, tid_own, n, gidlow, params,
             mc_table, dst_offset);
  PVK_CHECK_LAUNCH("pvk_segment_rename_mcast");
  return PVK_OK;
}
