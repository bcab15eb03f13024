// pvk_resynth.cu -- phase-preserving sum-of-sinusoids resynthesis for sm_100a
// (SinSum.synth -> RegPartial.synth, PVAnalysis.py:1053-1070,684-756).
//
// One CTA owns one output block of `hop` samples.  Every hop-block of a partial depends on
// at most 4 neighbouring f, 3 mag and 2 realph values of that partial and the reference's
// cumsum never crosses a block (:703-736), so blocks are independent (SURVEY appendix A6).
// The CTA turns the partials of its own frame row into closed-form coefficients staged in
// shared memory -- the phase of a block is a piecewise quadratic of the sample index because
// the frequency is piecewise linear with one knot per block -- and renders them: fp64 phase
// polynomial in cycles once per chunk of consecutive samples, exact range reduction, fp32
// quadratic + one MUFU cosine per partial-sample.  Fade-in heads / fade-out tails come from
// the +-ceil(E/hop) neighbour rows; a per-row flag (resynth_flags_kernel) says which of them
// hold the first / last frame of a rendered partial, the others are never touched.
// Not HBM bound (8 bytes written per output sample, ~0.03-0.1 B per partial-sample): the
// binding resources are MUFU and instruction issue; see DESIGN.md.
// Integrated-phase mode (phase_preserve = 0, pvk_resynth_ex): the phase runs on over the whole
// partial instead of being re-anchored at realph every block, so the start phase of each block is
// computed first by a segmented scan over the packed points (phase_scan_*); the render kernels are
// the same, instantiated with FREE = true (DESIGN.md 4.3).
#include "pvk_common.cuh"

namespace pvk {

struct RParams {
  const int32_t *tid;       // [F, K]
  const int32_t *tstart, *tlen;
  const int64_t *toff;
  const double *pf, *pmag, *prealph;
  int64_t F;
  int64_t ntcap;            // capacity of tstart / tlen / toff: ids at or beyond it are ignored (a caller that
                            // sized them by an upper bound which turned out too small renders again, sized exactly)
  int K;
  double sr, fstep, dfr;
  int h;                    // synthesis hop
  int E;                    // int(dfr*hop*edge)  (:740, :1056)
  float einv;               // 1 / E
  int dE;                   // ceil(E / h)
  int minframes;
  double *out;
  int64_t nout, block0;
  const uint32_t *mask;     // [F][2][mwk] slots holding the first (0) / last (1) frame of a rendered partial
  const struct TrackFade *tfade;   // [ntracks] fade-in / fade-out parameters of the rendered partials
  const struct BodyItem *gitems;   // [chunk blocks][K] staged partial bodies of the chunk's rows
  const int32_t *gcount;    // [chunk blocks] valid entries per row of gitems
  int64_t chunk0;           // first block of the chunk gitems / gcount describe
  int mwk;                  // mask words per row and kind, ceil(K / 32)
  int qk, qkm;              // knot of the frequency / amplitude interpolation inside a block
  int Af, Am;               // floor of the knot offsets dfr + 0.5 (:701) and dfr (:702)
  double qaf, qam;          // fractional knot offsets times h (qk = ceil(qaf), qkm = ceil(qam))
  double inv_sr, inv_h, hpc;   // 1/sr, 1/h, pi / (2 fstep) (:715)
  int nchp, G;              // chunk threads per item group, number of item groups
  // integrated-phase mode (phase_preserve = 0) only
  unsigned long long *phase;   // [phcap] start phase of every packed point's body block, fixed point (PHASE_ONE)
  int64_t phcap;            // capacity of phase: partials with points at or beyond it are not rendered
  double fscale;            // frequency ratio
  int free_phase;           // 1: integrated phase (launch-uniform; the render kernels take it as a template)
  const double *fcurve;     // [F] frequency ratio of every table row, in place of fscale (NULL: fscale;
                            // launch-uniform, the kernels take it as the template flag CURVE)
  int64_t fcurve_len;       // rows fcurve covers (checked >= F on the host).  With it RParams grows by 16
                            // bytes, so the kernel arguments after it keep their 16-byte alignment and the
                            // scalar-ratio kernels compile to the same instructions as without a curve
};

// np.interp at knot coordinate kf (sample position / h - knot offset) of values v[0..nfr),
// clamped at both ends like np.interp (:701-702)
__device__ __forceinline__ double lerp_knots(const double *__restrict__ v, int nfr, double kf) {
  if (!(kf > 0.0)) return v[0];
  if (kf >= (double)(nfr - 1)) return v[nfr - 1];
  int j = (int)kf;
  if (j > nfr - 2) j = nfr - 2;
  return fma(v[j + 1] - v[j], kf - (double)j, v[j]);
}

// value(q) on block ii, q in [0,h]: q < qk ? c0 + s0*q : c1 + s1*q, where the knot k0 = ii - A of
// the interpolated series sits at q = qa = alpha*h inside the block (a = A + alpha, :701-702)
struct Lin2 { double c0, s0, c1, s1; };

__device__ __forceinline__ Lin2 interp_block(const double *__restrict__ v, int nfr, int k0, double qa, double h,
                                             double inv_h) {
  Lin2 L;
  // segment 0: between knots k0-1 and k0
  if (k0 <= 0) { L.c0 = v[0]; L.s0 = 0.0; }
  else if (k0 - 1 >= nfr - 1) { L.c0 = v[nfr - 1]; L.s0 = 0.0; }
  else {
    const double slope = (v[k0] - v[k0 - 1]) * inv_h;
    L.c0 = v[k0 - 1] + slope * (h - qa); L.s0 = slope;
  }
  // segment 1: between knots k0 and k0+1
  if (k0 < 0) { L.c1 = v[0]; L.s1 = 0.0; }
  else if (k0 >= nfr - 1) { L.c1 = v[nfr - 1]; L.s1 = 0.0; }
  else {
    const double slope = (v[k0 + 1] - v[k0]) * inv_h;
    L.c1 = v[k0] - slope * qa; L.s1 = slope;
  }
  return L;
}

// sum_{u<q} F(u) of the piecewise linear F with its knot at sample qk
__device__ __forceinline__ double cum_sum(const Lin2 &L, double qk, double q) {
  const double qe = fmin(qk, q);
  const double te = qe * (qe - 1.0), tq = q * (q - 1.0);
  return (L.c0 * qe + 0.5 * L.s0 * te) + (L.c1 * (q - qe) + 0.5 * L.s1 * (tq - te));
}

// A partial body inside one block: two segments (before / after the block's knot) of the phase
// polynomial theta(q) = A + B q + C q^2 (cycles) and of the linear amplitude mc + ms q.  The
// knots qk (phase) and qkm (amplitude) depend on nfft/hop_an only, i.e. they are the same for
// every partial of a launch, so a thread picks its segment once, outside the item loop.
// tB = 2 pi B and tC2 = 4 pi C are the fp32 slope terms of the per-chunk quadratic.
struct __align__(16) PhaseSeg {
  double A, B;
  double C; float tB, tC2;
};
struct __align__(16) BodyItem {                                   // 80 bytes
  PhaseSeg s[2];
  float mc0, ms0, mc1, ms1;
};

// fade-in head (PVAnalysis.py:740-745) and fade-out tail (:748-751) of a rendered partial:
// constant frequency (cycles per sample) and amplitude under a raised cosine.  thh = phase of
// the first body sample, thl = phase of the last body sample, in cycles.
struct __align__(16) TrackFade {
  double thh, fch, thl, fct;
  float m0h, m0t; int pad0, pad1;
};                                                                // 48 bytes

constexpr double INV_2PI = 0.15915494309189535;
constexpr double TWO_PI = 6.283185307179586;


// Fractional part of a phase `th` (cycles, |th| < 2^28) as an fp32 angle in [0, 2 pi): adding
// 1.5 * 2^29 leaves round(th * 2^23) mod 2^23 in the low mantissa bits (exact reduction mod 1, rounded
// to 2^-23 cycles = 7.5e-7 rad), which become the mantissa of a float in [2^23, 2^24); one DADD, one
// LOP3 and one FFMA -- no fp64 -> fp32 conversion (a quarter-rate XU instruction next to the MUFUs).
__device__ __forceinline__ float frac_angle(double th) {
  const unsigned lo = (unsigned)__double_as_longlong(th + 805306368.0);
  const float x = __uint_as_float((lo & 0x7fffffu) | 0x4b000000u);
  return fmaf(x, 7.4901405e-7f, -6.2831855f);                    // (x - 2^23) * 2 pi / 2^23
}

// Integrated phase is kept as a 63-bit fixed-point fraction of a cycle: adding two of them modulo
// PHASE_ONE is exact, hence associative, so the segmented scan of the block increments gives the
// same bits whatever the grouping of its sums (batch = per clip, chunked = one shot).
typedef unsigned long long phase_t;
constexpr phase_t PHASE_MASK = 0x7fffffffffffffffull;        // PHASE_ONE - 1, PHASE_ONE = 2^63
constexpr phase_t PHASE_HEAD = 0x8000000000000000ull;        // flag bit of the scan's group aggregates

__device__ __forceinline__ phase_t phase_fix(double cyc) {
  const double fr = cyc - floor(cyc);                           // [0, 1]
  return (phase_t)(fr * 9.223372036854775808e18) & PHASE_MASK;   // * 2^63
}
__device__ __forceinline__ double phase_cycles(phase_t u) {
  return (double)(u & PHASE_MASK) * 1.0842021724855044e-19;    // * 2^-63
}

// frequency ratio of table row `row`: the launch's fscale, or the curve's value of that row (CURVE)
template <bool CURVE>
__device__ __forceinline__ double row_ratio(const RParams &p, int64_t row) {
  return CURVE ? p.fcurve[row] : p.fscale;
}

// body of partial v (nfr frames) inside block b, in cycles.  FREE = false: phase-preserving
// (PVAnalysis.py:701-736); FREE = true: integrated phase, starting at the scanned P of the block,
// frequency scaled by fscale (CURVE: by the curve's ratio of row b), no per-block correction (DESIGN.md 4.3)
template <bool FREE, bool CURVE>
__device__ __forceinline__ void make_body(const RParams &p, int64_t b, int v, int nfr, BodyItem &it) {
  const double h = (double)p.h;
  const int ii = (int)(b - p.tstart[v]);
  const int64_t o = p.toff[v];
  const double *tf = p.pf + o, *tm = p.pmag + o, *tr = p.prealph + o;
  const int k0 = ii - p.Af;
  const Lin2 Lf = interp_block(tf, nfr, k0, p.qaf, h, p.inv_h);
  const double qk = (double)p.qk;
  if (FREE) {
    const double fs = row_ratio<CURVE>(p, b) * p.inv_sr;
    const double th0 = phase_cycles(p.phase[o + ii]);
    const Lin2 Lm = interp_block(tm, nfr, ii - p.Am, p.qam, h, p.inv_h);
    PhaseSeg &s0 = it.s[0], &s1 = it.s[1];
    s0.A = th0;
    s0.B = (Lf.c0 - 0.5 * Lf.s0) * fs;
    s0.C = 0.5 * Lf.s0 * fs;
    s1.A = th0 + ((Lf.c0 - Lf.c1) * qk + 0.5 * (Lf.s0 - Lf.s1) * (qk * (qk - 1.0))) * fs;
    s1.B = (Lf.c1 - 0.5 * Lf.s1) * fs;
    s1.C = 0.5 * Lf.s1 * fs;
    s0.tB = (float)(TWO_PI * s0.B); s0.tC2 = (float)(2.0 * TWO_PI * s0.C);
    s1.tB = (float)(TWO_PI * s1.B); s1.tC2 = (float)(2.0 * TWO_PI * s1.C);
    it.mc0 = (float)Lm.c0; it.ms0 = (float)Lm.s0;
    it.mc1 = (float)Lm.c1; it.ms1 = (float)Lm.s1;
    return;
  }
  const double fb0 = p.qk > 0 ? Lf.c0 : Lf.c1;                      // fsig[hop*ii]
  const double fb1 = fma(Lf.s1, h, Lf.c1);                          // fsig[hop*(ii+1)]
  const double ph0 = tr[ii] + (fb1 - fb0) * p.hpc;                  // realph[ii] + phcor  :715,721
  const double th0 = ph0 * INV_2PI;
  double dphc = 0.0;
  if (ii < nfr - 1) {
    double fb2;                                                     // fsig[hop*(ii+2)]
    const int k1 = k0 + 1;
    if (k1 < 0) fb2 = tf[0];
    else if (k1 >= nfr - 1) fb2 = tf[nfr - 1];
    else fb2 = tf[k1] + (tf[k1 + 1] - tf[k1]) * p.inv_h * (h - p.qaf);
    const double phn = tr[ii + 1] + (fb2 - fb1) * p.hpc;            // realph[ii+1] + phcornext :717-718
    // phend = ph[-1] + 2 pi fsig[hop*(ii+1)]/sr (:726); dph = mod(phn - phend + pi, 2 pi) - pi (:727)
    const double xc = (phn - ph0) * INV_2PI - (cum_sum(Lf, qk, h - 1.0) + fb1) * p.inv_sr + 0.5;
    dphc = (xc - floor(xc) - 0.5) * p.inv_h;                        // :728-729, cycles per sample
  }
  const Lin2 Lm = interp_block(tm, nfr, ii - p.Am, p.qam, h, p.inv_h);
  PhaseSeg &s0 = it.s[0], &s1 = it.s[1];
  s0.A = th0;
  s0.B = (Lf.c0 - 0.5 * Lf.s0) * p.inv_sr + dphc;
  s0.C = 0.5 * Lf.s0 * p.inv_sr;
  s1.A = th0 + ((Lf.c0 - Lf.c1) * qk + 0.5 * (Lf.s0 - Lf.s1) * (qk * (qk - 1.0))) * p.inv_sr;
  s1.B = (Lf.c1 - 0.5 * Lf.s1) * p.inv_sr + dphc;
  s1.C = 0.5 * Lf.s1 * p.inv_sr;
  s0.tB = (float)(TWO_PI * s0.B); s0.tC2 = (float)(2.0 * TWO_PI * s0.C);
  s1.tB = (float)(TWO_PI * s1.B); s1.tC2 = (float)(2.0 * TWO_PI * s1.C);
  it.mc0 = (float)Lm.c0; it.ms0 = (float)Lm.s0;
  it.mc1 = (float)Lm.c1; it.ms1 = (float)Lm.s1;
}

// ------------------------------------------------------------------ kernel 1: per partial
// One warp per partial.  For the rendered ones (tlen >= minframes, :1061): find the slots of the
// first and the last frame in the frame table, set their bits in the start / end masks and store
// the fade-in / fade-out parameters.  CURVE: the head runs at the ratio of the first row, the tail at
// the ratio of the last row.
template <bool CURVE>
__global__ void __launch_bounds__(256) resynth_tracks_kernel(RParams p, int64_t ntracks,
                                                             const int32_t *__restrict__ ntracks_dev,
                                                             uint32_t *__restrict__ mask, TrackFade *__restrict__ tfade) {
  const int lane = threadIdx.x & 31;
  if (ntracks_dev != nullptr) { const int64_t m = *ntracks_dev; ntracks = m < ntracks ? m : ntracks; }
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < ntracks; v += nw) {
    const int nfr = p.tlen[v];
    if (nfr < p.minframes || nfr <= 0) continue;
    const int64_t s = p.tstart[v], e = s + nfr - 1;
    if (s < 0 || e >= p.F) continue;
    if (p.free_phase) {
      // Nyquist rule (flag set by the scan) or points beyond the phase buffer: not rendered; the flag
      // (tfade[v].pad0 != 0) takes the partial out of the render kernels' `on` predicate
      if (tfade[v].pad0 != 0 || p.toff[v] + nfr > p.phcap) {
        if (lane == 0) tfade[v].pad0 = 1;
        continue;
      }
    }
    for (int c0 = 0; c0 < p.K; c0 += 32) {
      const int c = c0 + lane;
      const bool hs = c < p.K && p.tid[s * p.K + c] == (int)v;
      const bool he = c < p.K && p.tid[e * p.K + c] == (int)v;
      if (hs) atomicOr(&mask[(s * 2 + 0) * p.mwk + (c >> 5)], 1u << (c & 31));
      if (he) atomicOr(&mask[(e * 2 + 1) * p.mwk + (c >> 5)], 1u << (c & 31));
    }
    if (lane == 0) {
      const int64_t o = p.toff[v];
      const double *tf = p.pf + o, *tm = p.pmag + o, *tr = p.prealph + o;
      const double hd = (double)p.h;
      TrackFade t;
      t.thh = tr[0] * INV_2PI;                                      // realph[0] :745
      t.fch = tf[0] * p.inv_sr;
      t.m0h = (float)lerp_knots(tm, nfr, -p.dfr);                   // msig[0] :742
      const int il = nfr - 1;
      const Lin2 Lf = interp_block(tf, nfr, il - p.Af, p.qaf, hd, p.inv_h);
      const double fb0 = p.qk > 0 ? Lf.c0 : Lf.c1;
      const double fb1 = fma(Lf.s1, hd, Lf.c1);
      if (p.free_phase) {
        // integrated phase: theta(h*nfr - 1) = P of the last block + the scaled in-block sum
        const double fs = row_ratio<CURVE>(p, e) * p.inv_sr;
        t.fch *= row_ratio<CURVE>(p, s);
        t.thl = phase_cycles(p.phase[o + il]) + cum_sum(Lf, (double)p.qk, hd - 1.0) * fs;
        t.fct = tf[il] * fs;
      } else {
        t.thl = (tr[il] + (fb1 - fb0) * p.hpc) * INV_2PI + cum_sum(Lf, (double)p.qk, hd - 1.0) * p.inv_sr;   // ph[-1] :750
        t.fct = tf[il] * p.inv_sr;
      }
      t.m0t = (float)lerp_knots(tm, nfr, (double)nfr - p.dfr);      // msig[hop*nfr] :748
      t.pad0 = t.pad1 = 0;
      tfade[v] = t;
    }
  }
}

// ------------------------------------------------------------------ integrated phase: block start phases
// P[i] of packed point i = body block ii of partial v (i = toff[v] + ii): the phase, in cycles mod 1, of
// the block's first sample, realph[0] / 2 pi + sum_{j < ii} fscale * cum_sum(Lf_j, qk, h) / sr.  A
// segmented scan over the packed array (a segment per partial) in three passes, so that a partial of
// millions of frames is spread over the whole GPU: groups of SCAN_GROUP consecutive points (group
// sums + in-group scan), one CTA over the group sums, fix-up of the points before a group's first
// partial start.  The sums are exact (phase_t), so P depends on nothing but the partial's own points.
constexpr int SCAN_GROUP = 1024;                                  // points per group: 32 steps of one warp
constexpr int SCAN_CARRY_THREADS = 1024;
constexpr int SCAN_CARRY_SMEM = (SCAN_CARRY_THREADS / 32) * (int)(sizeof(unsigned long long) + sizeof(int));

// number of real packed points: toff[ntracks] (ntracks from the device when given), at most phcap
__device__ __forceinline__ int64_t scan_npoints(const RParams &p, int64_t &ntracks, const int32_t *ntracks_dev) {
  if (ntracks_dev != nullptr) { const int64_t m = *ntracks_dev; ntracks = m < ntracks ? m : ntracks; }
  if (ntracks <= 0) return 0;
  const int64_t n = p.toff[ntracks];
  return n < p.phcap ? n : p.phcap;
}

// partial holding packed point i: the largest v < ntracks with toff[v] <= i
__device__ __forceinline__ int64_t scan_find(const RParams &p, int64_t ntracks, int64_t i) {
  int64_t lo = 0, hi = ntracks - 1;
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) >> 1;
    if (p.toff[mid] <= i) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// fscale (CURVE: the ratio of row tstart[v] + j) * (phase advance over body block j of partial v),
// cycles mod 1
template <bool CURVE>
__device__ __forceinline__ phase_t block_advance(const RParams &p, int64_t v, int64_t j) {
  const int64_t o = p.toff[v];
  const Lin2 Lf = interp_block(p.pf + o, p.tlen[v], (int)j - p.Af, p.qaf, (double)p.h, p.inv_h);
  const double r = row_ratio<CURVE>(p, p.tstart[v] + j);
  return phase_fix(cum_sum(Lf, (double)p.qk, (double)p.h) * (r * p.inv_sr));
}

// pass 1: one warp per group, 32 consecutive points per step.  Element of point i: the head value
// realph[0] / 2 pi (flagged) when i starts its partial, else the advance of block i - 1.  Writes the
// in-group segmented inclusive scan; the group's last point also carries PHASE_HEAD when the group
// holds a partial start.  Points of partials above the Nyquist limit flag them in tfade[v].pad0 (CURVE:
// each point tested at the ratio of its own row).
template <bool CURVE>
__global__ void __launch_bounds__(256) phase_scan_groups_kernel(RParams p, int64_t ntracks,
                                                                const int32_t *__restrict__ ntracks_dev,
                                                                TrackFade *__restrict__ tfade) {
  const int lane = threadIdx.x & 31;
  const int64_t npts = scan_npoints(p, ntracks, ntracks_dev);
  const int64_t ngroups = (npts + SCAN_GROUP - 1) / SCAN_GROUP;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const double nyq = 0.5 * p.sr;
  for (int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; c < ngroups; c += nw) {
    const int64_t base = c * SCAN_GROUP;
    const int64_t last = (base + SCAN_GROUP < npts ? base + SCAN_GROUP : npts) - 1;
    // advance of the block before the group's first point (lane 31 of "step -1"); every lane then
    // walks forward from the partial of the group's first point (one search per group)
    int64_t v = scan_find(p, ntracks, base);
    phase_t dprev = base > p.toff[v] ? block_advance<CURVE>(p, v, base - 1 - p.toff[v]) : 0;
    int64_t vflag = -1;                                            // last partial this lane flagged
    phase_t carry = 0;
    bool seen = false;                                             // a partial start in the group so far
    for (int64_t s0 = base; s0 <= last; s0 += 32) {
      const int64_t i = s0 + lane;
      const bool valid = i <= last;
      phase_t d = 0, e = 0;
      bool head = false;
      if (valid) {
        while (p.toff[v + 1] <= i) ++v;
        const int64_t j = i - p.toff[v];
        head = j == 0;
        d = block_advance<CURVE>(p, v, j);
        const double r = row_ratio<CURVE>(p, p.tstart[v] + j);
        if (r * p.pf[i] >= nyq && v != vflag) {                    // one flag per lane and partial: the
          vflag = v;                                               // points of a skipped partial would
          if (tfade[v].pad0 == 0) atomicOr(&tfade[v].pad0, 1);     // otherwise all hit one word
        }
      }
      phase_t dup = __shfl_up_sync(FULL, d, 1);
      if (lane == 0) dup = dprev;
      dprev = __shfl_sync(FULL, d, 31);
      if (valid) e = head ? phase_fix(p.prealph[i] * INV_2PI) : dup;
      if (lane == 0 && !head) e = (e + carry) & PHASE_MASK;
      bool f = head;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {                           // segmented inclusive scan
        const phase_t eu = __shfl_up_sync(FULL, e, o);
        const bool fu = __shfl_up_sync(FULL, (int)f, o) != 0;
        if (lane >= o) {
          if (!f) e = (e + eu) & PHASE_MASK;
          f = f || fu;
        }
      }
      if (valid) p.phase[i] = (i == last && (seen || f)) ? (e | PHASE_HEAD) : e;
      carry = __shfl_sync(FULL, e, 31);
      seen = seen || __shfl_sync(FULL, (int)f, 31) != 0;
    }
  }
}

// pass 2: one CTA; thread t owns a contiguous run of groups.  Turns every group's last point into
// its final P (the carry of all earlier groups added up to the group's first partial start).
__global__ void __launch_bounds__(SCAN_CARRY_THREADS) phase_scan_carry_kernel(RParams p, int64_t ntracks,
                                                                              const int32_t *__restrict__ ntracks_dev) {
  PVK_SMEM(smem);                                                  // warp totals: SCAN_CARRY_SMEM bytes
  phase_t *s_val = reinterpret_cast<phase_t *>(smem);
  int *s_flag = reinterpret_cast<int *>(smem + (SCAN_CARRY_THREADS / 32) * sizeof(phase_t));
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const int64_t npts = scan_npoints(p, ntracks, ntracks_dev);
  const int64_t ngroups = (npts + SCAN_GROUP - 1) / SCAN_GROUP;
  const int64_t per = (ngroups + SCAN_CARRY_THREADS - 1) / SCAN_CARRY_THREADS;
  const int64_t g0 = t * per, g1 = g0 + per < ngroups ? g0 + per : ngroups;
  auto last_of = [&](int64_t c) { const int64_t e = (c + 1) * SCAN_GROUP; return (e < npts ? e : npts) - 1; };
  // this thread's aggregate
  phase_t a = 0;
  bool fa = false;
  for (int64_t c = g0; c < g1; ++c) {
    const phase_t x = p.phase[last_of(c)];
    if (x & PHASE_HEAD) { a = x & PHASE_MASK; fa = true; } else a = (a + x) & PHASE_MASK;
  }
  // exclusive segmented scan of the thread aggregates: warp, then the warp totals
  phase_t e = a;
  bool f = fa;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const phase_t eu = __shfl_up_sync(FULL, e, o);
    const bool fu = __shfl_up_sync(FULL, (int)f, o) != 0;
    if (lane >= o) {
      if (!f) e = (e + eu) & PHASE_MASK;
      f = f || fu;
    }
  }
  if (lane == 31) { s_val[w] = e; s_flag[w] = f ? 1 : 0; }
  __syncthreads();
  phase_t wcarry = 0;                                             // inclusive total of the warps before w
  for (int k = 0; k < w; ++k) wcarry = s_flag[k] ? s_val[k] : (wcarry + s_val[k]) & PHASE_MASK;
  phase_t ex = __shfl_up_sync(FULL, e, 1);                        // inclusive total of the lanes before
  bool fex = __shfl_up_sync(FULL, (int)f, 1) != 0;
  if (lane == 0) { ex = 0; fex = false; }
  phase_t run = fex ? ex : (wcarry + ex) & PHASE_MASK;
  for (int64_t c = g0; c < g1; ++c) {
    const int64_t l = last_of(c);
    const phase_t x = p.phase[l];
    run = (x & PHASE_HEAD) ? (x & PHASE_MASK) : (run + x) & PHASE_MASK;
    p.phase[l] = run;
  }
}

// pass 3: one warp per group c > 0: the points before the group's first partial start (all but the
// last point, final since pass 2) get the final P of the previous group's last point added.
__global__ void __launch_bounds__(256) phase_scan_fixup_kernel(RParams p, int64_t ntracks,
                                                               const int32_t *__restrict__ ntracks_dev) {
  const int lane = threadIdx.x & 31;
  const int64_t npts = scan_npoints(p, ntracks, ntracks_dev);
  const int64_t ngroups = (npts + SCAN_GROUP - 1) / SCAN_GROUP;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t c = 1 + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); c < ngroups; c += nw) {
    const int64_t base = c * SCAN_GROUP;
    const int64_t last = (base + SCAN_GROUP < npts ? base + SCAN_GROUP : npts) - 1;
    const int64_t v0 = scan_find(p, ntracks, base);
    if (p.toff[v0] == base) continue;                              // the group starts a partial
    const int64_t stop = p.toff[v0 + 1] < last ? p.toff[v0 + 1] : last;
    const phase_t carry = p.phase[base - 1];
    for (int64_t i = base + lane; i < stop; i += 32) p.phase[i] = (p.phase[i] + carry) & PHASE_MASK;
  }
}

// ------------------------------------------------------------------ kernel 2: per frame row
// One warp per row of the chunk: the bodies of the rendered partials of the row, as closed-form
// coefficients, compacted in slot order (deterministic sum order) into gitems.
template <bool FREE, bool CURVE>
__global__ void __launch_bounds__(128) resynth_prepare_kernel(RParams p, int64_t nrows, BodyItem *__restrict__ gitems,
                                                              int32_t *__restrict__ gcount) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= nrows) return;
  const int64_t b = p.chunk0 + row;
  int n = 0;
  if (b < p.F) {
    for (int c0 = 0; c0 < p.K; c0 += 32) {
      const int c = c0 + lane;
      int v = -1, nfr = 0;
      if (c < p.K) {
        v = p.tid[b * p.K + c];
        if (v >= 0 && v < p.ntcap) nfr = p.tlen[v];
      }
      const bool on = v >= 0 && nfr >= p.minframes && (!FREE || p.tfade[v].pad0 == 0);   // :1061; Nyquist rule
      const unsigned mk = __ballot_sync(FULL, on);
      if (on) make_body<FREE, CURVE>(p, b, v, nfr, gitems[row * p.K + n + __popc(mk & lanemask_lt())]);
      n += __popc(mk);
    }
  }
  if (lane == 0) gcount[row] = n;
}

// ------------------------------------------------------------------ kernel 3: render
// Inner loops shared by the two render kernels.  A thread owns RS consecutive samples qs..qs+RS
// of block b and adds the staged partial bodies items[c], c = g, g+G, ... < nbody, to acc[].
// Fast path (no knot inside the chunk -- practically always): the phase polynomial is evaluated
// once in fp64 at the chunk centre, reduced to an angle in [0, 2 pi) (frac_angle) and advanced over
// the RS samples as an fp32 quadratic in radians (|increment| < RS/2 * pi, so the MUFU cosine sees
// arguments in (-RS/2 * pi, 2 pi + RS/2 * pi), about +-30 rad at RS = 16); one MUFU cosine + 5 FMA-pipe
// instructions per partial-sample.  Slow path (knot inside the chunk): fp64 phase per sample.
template <int RS>
__device__ __forceinline__ void render_bodies(const RParams &p, const BodyItem *items, int nbody, int g, int G,
                                              int qs, bool fast, float *acc) {
  const float TWO_PI_F = 6.283185307179586f;
  if (fast) {
    const int sf = qs >= p.qk ? 1 : 0, sm = qs >= p.qkm ? 1 : 0;
    const double qcd = (double)(qs + RS / 2);
    const float qcf = (float)(qs + RS / 2);
    for (int c = g; c < nbody; c += G) {
      const PhaseSeg *sp = &items[c].s[sf];
      const double2 ab = *reinterpret_cast<const double2 *>(&sp->A);
      const double2 cw = *reinterpret_cast<const double2 *>(&sp->C);        // C | (tB, tC2)
      const float2 am = *reinterpret_cast<const float2 *>(&items[c].mc0 + 2 * sm);
      const float tB = __int_as_float((int)(__double_as_longlong(cw.y) & 0xffffffffLL));
      const float tC2 = __int_as_float((int)(__double_as_longlong(cw.y) >> 32));
      const double th = fma(fma(cw.x, qcd, ab.y), qcd, ab.x);     // cycles at the chunk centre
      const float t0 = frac_angle(th);                            // exact reduction mod 1 cycle
      const float t1 = fmaf(tC2, qcf, tB);
      const float t2 = 0.5f * tC2;
      const float a0 = fmaf(am.y, qcf, am.x);
#pragma unroll
      for (int m = 0; m < RS; ++m) {
        const float fm = (float)(m - RS / 2);
        const float cs = __cosf(fmaf(fmaf(t2, fm, t1), fm, t0));
        acc[m] = fmaf(fmaf(am.y, fm, a0), cs, acc[m]);
      }
    }
  } else {
    for (int c = g; c < nbody; c += G) {
#pragma unroll
      for (int m = 0; m < RS; ++m) {
        const int q = qs + m;
        if (q < p.h) {
          const PhaseSeg &sp = items[c].s[q >= p.qk ? 1 : 0];
          const float *sa = &items[c].mc0 + (q >= p.qkm ? 2 : 0);
          const double qd = (double)q;
          const double th = fma(fma(sp.C, qd, sp.B), qd, sp.A);
          const float fr = (float)(th - rint(th));
          acc[m] = fmaf(fmaf(sa[1], (float)q, sa[0]), __cosf(TWO_PI_F * fr), acc[m]);
        }
      }
    }
  }
}

// Fade-in heads of partials starting in rows (b, b+dE] and fade-out tails of partials ending in
// rows [b-dE, b): the start / end masks name the slots; no staging, no barrier.  The fades found
// are dealt round-robin to the G item groups (active: this thread renders at all).
template <int RS>
__device__ __forceinline__ void render_fades(const RParams &p, int64_t b, int qs, bool active, int g, int G,
                                             float *acc) {
  const float TWO_PI_F = 6.283185307179586f;
  const int K = p.K, h = p.h;
  int nf = 0;
  for (int64_t r = b - p.dE; r <= b + p.dE; ++r) {
    if (r == b || r < 0 || r >= p.F) continue;                  // uniform
    const bool head = r > b;
    const uint32_t *mw = p.mask + (r * 2 + (head ? 0 : 1)) * p.mwk;
    for (int w = 0; w < p.mwk; ++w) {
      uint32_t bits = mw[w];                                      // uniform
      while (bits) {
        const int c = w * 32 + __ffs((int)bits) - 1;
        bits &= bits - 1;
        const bool mine = active && (G == 1 || (nf % G) == g);
        ++nf;
        if (!mine) continue;
        const int v = p.tid[r * K + c];
        const TrackFade tf = p.tfade[v];
        double A, B;
        float m0;
        int qa, qb, eoff;
        if (head) {
          // head sample qh = q + off, off = (b - r)*h + E; valid 0 <= qh < E   (:740-745)
          const int64_t off = (b - r) * h + p.E;
          B = tf.fch; A = tf.thh - B * (double)((int64_t)p.E - off); m0 = tf.m0h;
          qa = (int)(off < 0 ? -off : 0); qb = h; eoff = (int)off;
        } else {
          // tail sample qt = q + off, off = (b - r - 1)*h; valid 0 <= qt < E   (:748-751)
          const int64_t off = (b - r - 1) * h;
          B = tf.fct; A = tf.thl + B * (double)(off + 1); m0 = tf.m0t;
          const int64_t qe = (int64_t)p.E - off;
          qa = 0; qb = (int)(qe < h ? qe : h); eoff = (int)off;
        }
        if (qb <= qs || qa >= qs + RS) continue;
        if (qa <= qs && qs + RS <= qb) {
          // whole chunk inside the fade: linear phase and linear envelope angle in fp32
          const double qcd = (double)(qs + RS / 2);
          const double th = fma(B, qcd, A);
          const float t0 = frac_angle(th);
          const float t1 = TWO_PI_F * (float)B;
          const float e1 = 3.14159265358979f * p.einv;
          const float e0 = e1 * (float)(qs + RS / 2 + eoff);
          const float hm = 0.5f * m0, sg = head ? -hm : hm;      // m0 * (1 -+ cos) / 2
          if (e1 * (float)(RS / 2) <= 0.05f) {                   // (uniform: E is a launch parameter)
            // slow raised cosine (E >= ~500 samples): cubic Taylor polynomial of the envelope around the
            // chunk centre -- |x| <= 0.05 rad, remainder x^4/24 <= 2.6e-7 of the fade amplitude -- on the FMA
            // pipe; two MUFUs per chunk instead of one per sample (the XU pipe is what binds this kernel)
            const float c0 = __cosf(e0), s0 = __sinf(e0);
            const float a0 = fmaf(sg, c0, hm), a1 = -sg * s0 * e1, a2 = -0.5f * sg * c0 * e1 * e1;
            const float a3 = sg * s0 * e1 * e1 * e1 * (1.f / 6.f);
#pragma unroll
            for (int m = 0; m < RS; ++m) {
              const float fm = (float)(m - RS / 2);
              const float am = fmaf(fmaf(fmaf(a3, fm, a2), fm, a1), fm, a0);
              acc[m] = fmaf(am, __cosf(fmaf(t1, fm, t0)), acc[m]);
            }
          } else {
#pragma unroll
            for (int m = 0; m < RS; ++m) {
              const float fm = (float)(m - RS / 2);
              const float ce = __cosf(fmaf(e1, fm, e0));
              acc[m] = fmaf(fmaf(sg, ce, hm), __cosf(fmaf(t1, fm, t0)), acc[m]);
            }
          }
        } else {
#pragma unroll
          for (int m = 0; m < RS; ++m) {
            const int q = qs + m;
            if (q >= qa && q < qb) {
              const double th = fma(B, (double)q, A);
              const float fr = (float)(th - rint(th));
              const float ce = __cosf(3.14159265358979f * (float)(q + eoff) * p.einv);
              const float am = m0 * (head ? 0.5f * (1.f - ce) : 0.5f * (1.f + ce));
              acc[m] = fmaf(am, __cosf(TWO_PI_F * fr), acc[m]);
            }
          }
        }
      }
    }
  }
}

// General render kernel (any hop): one CTA renders one output block of h samples.  Thread
// t = g * nchp + ch: chunk ch (RS consecutive samples) of item group g; the groups split the
// partials of the block among themselves and their partial sums are added through shared memory.
template <int RS>
__global__ void __launch_bounds__(128, 8) resynth_kernel(RParams p) {
  PVK_SMEM(smem);
  const int K = p.K, h = p.h, BD = blockDim.x;
  BodyItem *items = reinterpret_cast<BodyItem *>(smem);
  float *red = reinterpret_cast<float *>(smem + (size_t)K * sizeof(BodyItem));
  const int RSTRIDE = BD + 32 / RS;
  const int tid = threadIdx.x;
  const int64_t b = p.block0 + blockIdx.x;
  const int64_t nbase = b * (int64_t)h;

  // ---- the staged partial bodies of row b: global -> shared, 16 bytes per thread and step
  const int nbody = p.gcount[b - p.chunk0];
  {
    const int4 *src = reinterpret_cast<const int4 *>(p.gitems + (b - p.chunk0) * K);
    int4 *dst = reinterpret_cast<int4 *>(items);
    const int n16 = nbody * (int)(sizeof(BodyItem) / 16);
    for (int i = tid; i < n16; i += BD) dst[i] = src[i];
  }
  __syncthreads();

  const int nchp = p.nchp, G = p.G, W = nchp * RS;
  const int g = tid / nchp, ch = tid - g * nchp;
  for (int q0 = 0; q0 < h; q0 += W) {
    const int qs = q0 + ch * RS;
    const bool active = g < G && qs < h;
    float acc[RS];
#pragma unroll
    for (int m = 0; m < RS; ++m) acc[m] = 0.f;
    const bool fast = (qs + RS <= h) && !(qs < p.qk && p.qk < qs + RS) && !(qs < p.qkm && p.qkm < qs + RS);
    if (active) render_bodies<RS>(p, items, nbody, g, G, qs, fast, acc);
    render_fades<RS>(p, b, qs, active, g, G, acc);

    // ---- add the groups' partial sums and write the block (coalesced fp64 stores)
    if (g < G) {
#pragma unroll
      for (int m = 0; m < RS; ++m) red[m * RSTRIDE + tid] = acc[m];
    }
    __syncthreads();
    for (int q = tid; q < W; q += BD) {
      const int64_t n = nbase + q0 + q;
      if (q0 + q < h && n < p.nout) {
        const int cq = q / RS, m = q - cq * RS;
        float s = 0.f;
        for (int gg = 0; gg < G; ++gg) s += red[m * RSTRIDE + gg * nchp + cq];
        p.out[n - p.block0 * (int64_t)h] = (double)s;
      }
    }
    __syncthreads();
  }
}

// Tile render kernel (hop a multiple of 32*RS): one WARP renders one tile of 32*RS consecutive
// samples of a block, lane l the samples [l*RS, (l+1)*RS).  No block barrier, no cross-group
// reduction, block-level scalar work (row lookup, fade scan) done once per tile.  The partial
// bodies are NOT staged in HBM: the warp walks the block's frame row 32 slots at a time, every
// lane turns the rendered partial of its slot into closed-form coefficients (make_body) and puts
// them, compacted in slot order (deterministic sum order), into the warp's shared-memory buffer,
// from which all lanes render them.  The slot ids of the next group are in flight while the current
// group is rendered; the dependent loads of make_body (track meta -> 9 table values) are hidden by
// the other resident warps.  The finished tile is transposed through the same buffer so that the
// fp64 stores are coalesced.
constexpr int TILE_BATCH = 32;
constexpr int TILE_WARP_BYTES = TILE_BATCH * (int)sizeof(BodyItem);   // 2560 >= RS * 33 * 4 for RS <= 16
constexpr int TILE_WARPS = 4;

template <int RS, bool FREE, bool CURVE>
__global__ void __launch_bounds__(TILE_WARPS * 32, 8) resynth_tile_kernel(RParams p, int64_t ntiles, int tpb) {
  PVK_SMEM(smem);
  constexpr int TILE = 32 * RS;
  static_assert(RS * 33 * 4 <= TILE_WARP_BYTES, "transpose buffer");
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t tile = (int64_t)blockIdx.x * TILE_WARPS + warp;
  if (tile >= ntiles) return;                                     // warp uniform; the kernel has no block barrier
  BodyItem *items = reinterpret_cast<BodyItem *>(smem + warp * TILE_WARP_BYTES);
  const int h = p.h, K = p.K;
  const int64_t b = p.block0 + tile / tpb;
  const int q0 = (int)(tile % tpb) * TILE;
  const int qs = q0 + lane * RS;

  float acc[RS];
#pragma unroll
  for (int m = 0; m < RS; ++m) acc[m] = 0.f;
  const bool fast = !(qs < p.qk && p.qk < qs + RS) && !(qs < p.qkm && p.qkm < qs + RS);

  if (b < p.F) {
    const int32_t *trow = p.tid + b * K;
    int vnext = lane < K ? trow[lane] : -1;
    for (int c0 = 0; c0 < K; c0 += 32) {
      const int v = vnext;
      const int cn = c0 + 32 + lane;
      vnext = cn < K ? trow[cn] : -1;
      const int nfr = (v >= 0 && v < p.ntcap) ? p.tlen[v] : 0;
      const bool on = v >= 0 && nfr >= p.minframes && (!FREE || p.tfade[v].pad0 == 0);   // :1061; Nyquist rule
      const unsigned mk = __ballot_sync(FULL, on);
      if (mk == 0u) continue;                                      // warp uniform
      if (on) make_body<FREE, CURVE>(p, b, v, nfr, items[__popc(mk & lanemask_lt())]);
      __syncwarp();
      render_bodies<RS>(p, items, __popc(mk), 0, 1, qs, fast, acc);
      __syncwarp();
    }
  }
  render_fades<RS>(p, b, qs, true, 0, 1, acc);

  // ---- transpose through shared memory, coalesced fp64 stores
  float *red = reinterpret_cast<float *>(items);
#pragma unroll
  for (int m = 0; m < RS; ++m) red[lane * (RS + 1) + m] = acc[m];
  __syncwarp();
  const int64_t n0 = b * (int64_t)h + q0;
  double *o = p.out + (n0 - p.block0 * (int64_t)h);
#pragma unroll
  for (int j = 0; j < RS; ++j) {
    const int q = j * 32 + lane;
    if (n0 + q < p.nout) o[q] = (double)red[q + q / RS];
  }
}

}  // namespace pvk

using namespace pvk;

static int64_t resynth_fixed_ws(int64_t nframes, int npks, int64_t ntracks) {
  const int64_t mwk = (npks + 31) / 32;
  return align_up(nframes * 2 * mwk * 4, 256) + align_up(ntracks * (int64_t)sizeof(TrackFade), 256);
}
static int64_t resynth_row_ws(int npks) { return (int64_t)npks * (int64_t)sizeof(BodyItem) + 4; }

// Scratch for pvk_resynth: start / end masks + fade parameters + staged bodies of up to
// 32768 blocks per chunk (larger block ranges are rendered chunk by chunk).
extern "C" int64_t pvk_resynth_workspace_bytes(int64_t nframes, int npks, int64_t ntracks, int64_t nblocks) {
  if (nframes < 0 || npks < 1 || ntracks < 0 || nblocks < 0) return -1;
  const int64_t cb = nblocks < 32768 ? (nblocks < 1 ? 1 : nblocks) : 32768;
  return resynth_fixed_ws(nframes, npks, ntracks) + align_up(cb * resynth_row_ws(npks), 256) + 512;
}

template <int RS>
static int launch_resynth(const RParams &p, int64_t nblocks, int bd, void *stream) {
  const int smem = p.K * (int)sizeof(BodyItem) + RS * (bd + 32 / RS) * 4;
  if (smem > 48 * 1024) {
    if (PVK_SET_SMEM(resynth_kernel<RS>, smem) != 0) {
      set_error("pvk_resynth: cannot reserve %d bytes of shared memory", smem);
      return PVK_ERR_CUDA;
    }
  }
  PVK_LAUNCH(resynth_kernel<RS>, dim3((unsigned)nblocks), dim3(bd), smem, stream, p);
  PVK_CHECK_LAUNCH("pvk_resynth(render)");
  return PVK_OK;
}

template <int RS>
static int launch_resynth_tile(const RParams &p, int64_t nblocks, void *stream) {
  const int tpb = p.h / (32 * RS);
  const int64_t ntiles = nblocks * tpb;
  const dim3 grid((unsigned)((ntiles + TILE_WARPS - 1) / TILE_WARPS)), block(TILE_WARPS * 32);
  if (p.fcurve != nullptr)
    PVK_LAUNCH((resynth_tile_kernel<RS, true, true>), grid, block, TILE_WARPS * TILE_WARP_BYTES, stream, p, ntiles, tpb);
  else if (p.free_phase)
    PVK_LAUNCH((resynth_tile_kernel<RS, true, false>), grid, block, TILE_WARPS * TILE_WARP_BYTES, stream, p, ntiles, tpb);
  else
    PVK_LAUNCH((resynth_tile_kernel<RS, false, false>), grid, block, TILE_WARPS * TILE_WARP_BYTES, stream, p, ntiles, tpb);
  PVK_CHECK_LAUNCH("pvk_resynth(render tiles)");
  return PVK_OK;
}

extern "C" int pvk_resynth(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks, const int32_t *tstart,
                           const int32_t *tlen, const int64_t *toff, const double *pf, const double *pmag,
                           const double *prealph, double sr, int hop, int nfft, int hop_an, double edge,
                           int minframes, double *out, int64_t nout, int64_t block0, int64_t nblocks,
                           void *workspace, int64_t workspace_bytes, int reuse_tracks, void *stream) {
  return pvk_resynth_dev(tid, nframes, npks, ntracks, nullptr, tstart, tlen, toff, pf, pmag, prealph, sr, hop, nfft, hop_an,
                         edge, minframes, out, nout, block0, nblocks, workspace, workspace_bytes, reuse_tracks, stream);
}

extern "C" int pvk_resynth_dev(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                               const int32_t *ntracks_dev, const int32_t *tstart, const int32_t *tlen,
                               const int64_t *toff, const double *pf, const double *pmag, const double *prealph,
                               double sr, int hop, int nfft, int hop_an, double edge, int minframes, double *out,
                               int64_t nout, int64_t block0, int64_t nblocks, void *workspace,
                               int64_t workspace_bytes, int reuse_tracks, void *stream) {
  return pvk_resynth_ex(tid, nframes, npks, ntracks, ntracks_dev, tstart, tlen, toff, pf, pmag, prealph, sr, hop, nfft,
                        hop_an, edge, minframes, out, nout, block0, nblocks, workspace, workspace_bytes, reuse_tracks,
                        1, 1.0, nullptr, 0, stream);
}

// sample rate, hops and knots of a launch (everything but the tables and the output)
static void synth_params(RParams &p, double sr, int hop, int nfft, int hop_an, int npks, double fscale) {
  p.K = npks; p.sr = sr;
  p.fstep = sr / (double)nfft;                               // :825
  const double overlap = (double)hop_an / (double)nfft;      // :824
  p.dfr = 1.0 / overlap / 2.0;                               // :687
  p.h = hop;
  {  // knots of the interpolated frequency (:701) / amplitude (:702) inside a block
    const double af = p.dfr + 0.5, am = p.dfr;
    p.Af = (int)floor(af); p.Am = (int)floor(am);
    p.qaf = (af - floor(af)) * (double)hop; p.qam = (am - floor(am)) * (double)hop;
    p.qk = (int)ceil(p.qaf); p.qkm = (int)ceil(p.qam);
  }
  p.inv_sr = 1.0 / sr; p.inv_h = 1.0 / (double)hop;
  p.hpc = 3.141592653589793 / (2.0 * p.fstep);
  p.mwk = (npks + 31) / 32;
  p.fscale = fscale;
  p.fcurve = nullptr;
  p.fcurve_len = 0;
}

// the argument checks of a frequency-ratio curve (the _curve exports): one ratio per table row, none
// together with a scalar ratio or the phase-preserving model; the values are the caller's to check
#define PVK_REQUIRE_CURVE(fn, nrows, phase_preserve)                                                            \
  do {                                                                                                       \
    if (fcurve != nullptr) {                                                                                 \
      PVK_REQUIRE(fcurve_len >= (nrows), fn ": fcurve_len=%lld is short (one ratio per frame row, %lld rows)", \
                  (long long)fcurve_len, (long long)(nrows));                                                \
      PVK_REQUIRE(fscale == 1.0, fn ": fscale=%g with an fcurve (the curve carries the ratio; pass 1)", fscale); \
      PVK_REQUIRE(!(phase_preserve), fn ": an fcurve needs phase_preserve=0 (the analysed phases do not fit a " \
                  "scaled frequency)");                                                                      \
    }                                                                                                        \
  } while (0)

// block start phases + Nyquist flags (tfade[v].pad0) of every partial: the three scan passes
static int launch_phase_scan(const RParams &p, int64_t ntracks, const int32_t *ntracks_dev, TrackFade *tfade,
                             void *stream) {
  cudaMemsetAsync(tfade, 0, (size_t)(ntracks * (int64_t)sizeof(TrackFade)), (cudaStream_t)stream);
  const int64_t pcap = p.phcap < p.F * (int64_t)p.K ? p.phcap : p.F * (int64_t)p.K;
  int64_t sg = ((pcap + SCAN_GROUP - 1) / SCAN_GROUP * 32 + 255) / 256;
  if (sg > 148 * 16) sg = 148 * 16;
  if (sg < 1) sg = 1;
  if (p.fcurve != nullptr)
    PVK_LAUNCH(phase_scan_groups_kernel<true>, dim3((unsigned)sg), dim3(256), 0, stream, p, ntracks, ntracks_dev, tfade);
  else
    PVK_LAUNCH(phase_scan_groups_kernel<false>, dim3((unsigned)sg), dim3(256), 0, stream, p, ntracks, ntracks_dev, tfade);
  PVK_CHECK_LAUNCH("pvk_resynth(phase scan)");
  PVK_LAUNCH(phase_scan_carry_kernel, dim3(1), dim3(SCAN_CARRY_THREADS), SCAN_CARRY_SMEM, stream, p, ntracks, ntracks_dev);
  PVK_CHECK_LAUNCH("pvk_resynth(phase carry)");
  PVK_LAUNCH(phase_scan_fixup_kernel, dim3((unsigned)sg), dim3(256), 0, stream, p, ntracks, ntracks_dev);
  PVK_CHECK_LAUNCH("pvk_resynth(phase fix-up)");
  return PVK_OK;
}

// pvk_resynth_ex (scan = true) and pvk_resynth_render (scan = false: the block start phases and the
// Nyquist flags are already in the workspace / phase_ws)
static int resynth_run(bool scan, const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                       const int32_t *ntracks_dev, const int32_t *tstart, const int32_t *tlen,
                       const int64_t *toff, const double *pf, const double *pmag, const double *prealph,
                       double sr, int hop, int nfft, int hop_an, double edge, int minframes, double *out,
                       int64_t nout, int64_t block0, int64_t nblocks, void *workspace,
                       int64_t workspace_bytes, int reuse_tracks, int phase_preserve, double fscale,
                       const double *fcurve, int64_t fcurve_len, double *phase_ws, int64_t phase_ws_len,
                       void *stream) {
  PVK_REQUIRE(isfinite(fscale) && fscale > 0.0, "pvk_resynth: fscale=%g must be finite and > 0", fscale);
  PVK_REQUIRE(!phase_preserve || fscale == 1.0,
              "pvk_resynth: fscale=%g needs phase_preserve=0 (the analysed phases do not fit a scaled frequency)",
              fscale);
  if (!phase_preserve) {
    // every partial has at least one point and there are at most nframes * npks points
    const int64_t need = ntracks < nframes * (int64_t)npks ? ntracks : nframes * (int64_t)npks;
    PVK_REQUIRE(phase_ws != nullptr, "pvk_resynth: phase_ws is NULL (phase_preserve=0 needs one double per packed point)");
    PVK_REQUIRE(phase_ws_len >= need,
                "pvk_resynth: phase_ws_len=%lld is short (one double per packed point, at least %lld)",
                (long long)phase_ws_len, (long long)need);
  }
  PVK_REQUIRE(hop >= 1 && nfft >= 1 && hop_an >= 1, "pvk_resynth: hop=%d nfft=%d hop_an=%d must be >= 1", hop, nfft, hop_an);
  PVK_REQUIRE(npks >= 1 && npks <= PVK_MAX_NPKS, "pvk_resynth: npks=%d must be in [1, %d]", npks, PVK_MAX_NPKS);
  PVK_REQUIRE(sr > 0.0 && edge >= 0.0, "pvk_resynth: sr and edge must be positive");
  PVK_REQUIRE(nout >= 0 && nframes >= 0 && block0 >= 0 && ntracks >= 0, "pvk_resynth: negative sizes");
  const int64_t nblk_total = (nout + hop - 1) / hop;
  if (nblocks < 0) nblocks = nblk_total - block0;
  if (nblocks <= 0 || nout == 0) return PVK_OK;
  PVK_REQUIRE(block0 + nblocks <= nblk_total, "pvk_resynth: block range [%lld, %lld) exceeds %lld blocks",
              (long long)block0, (long long)(block0 + nblocks), (long long)nblk_total);
  PVK_REQUIRE(out != nullptr, "pvk_resynth: out is NULL");
  PVK_REQUIRE(nframes == 0 || (tid && tstart && tlen && toff && pf && pmag && prealph),
              "pvk_resynth: NULL pointer argument");
  const int64_t fixed = resynth_fixed_ws(nframes, npks, ntracks);
  PVK_REQUIRE(workspace != nullptr && workspace_bytes >= fixed + align_up(resynth_row_ws(npks), 256) + 512,
              "pvk_resynth: workspace too small (%lld bytes; pvk_resynth_workspace_bytes gives the size)",
              (long long)workspace_bytes);
  RParams p;
  synth_params(p, sr, hop, nfft, hop_an, npks, fscale);
  p.tid = tid; p.tstart = tstart; p.tlen = tlen; p.toff = toff;
  p.pf = pf; p.pmag = pmag; p.prealph = prealph;
  p.F = nframes; p.ntcap = ntracks;
  p.E = (int)(p.dfr * (double)hop * edge);                   // :740
  p.dE = (p.E + hop - 1) / hop;
  p.einv = p.E > 0 ? (float)(1.0 / (double)p.E) : 0.f;
  p.minframes = minframes;
  p.out = out; p.nout = nout; p.block0 = block0;
  p.phase = reinterpret_cast<unsigned long long *>(phase_ws);
  p.phcap = phase_preserve ? 0 : phase_ws_len;
  p.free_phase = phase_preserve ? 0 : 1;
  p.fcurve = fcurve;
  p.fcurve_len = fcurve_len;

  // workspace: masks | fade parameters | staged bodies + counts of one chunk of blocks
  unsigned char *ws = reinterpret_cast<unsigned char *>(workspace);
  uint32_t *mask = reinterpret_cast<uint32_t *>(ws);
  const int64_t mask_bytes = align_up(nframes * 2 * p.mwk * 4, 256);
  TrackFade *tfade = reinterpret_cast<TrackFade *>(ws + mask_bytes);
  unsigned char *chunk_ws = ws + fixed;
  int64_t cb = (workspace_bytes - fixed - 512) / resynth_row_ws(npks);
  if (cb > nblocks) cb = nblocks;
  BodyItem *gitems = reinterpret_cast<BodyItem *>(chunk_ws);
  int32_t *gcount = reinterpret_cast<int32_t *>(chunk_ws + align_up(cb * npks * (int64_t)sizeof(BodyItem), 256));
  p.mask = mask; p.tfade = tfade; p.gitems = gitems; p.gcount = gcount;

  if (nframes > 0 && !reuse_tracks) cudaMemsetAsync(mask, 0, (size_t)(nframes * 2 * p.mwk * 4), (cudaStream_t)stream);
  if (ntracks > 0 && nframes > 0 && !reuse_tracks) {
    p.chunk0 = 0;
    if (p.free_phase && scan) {
      // block start phases + Nyquist flags (tfade[v].pad0), read by the tracks kernel below
      const int rc = launch_phase_scan(p, ntracks, ntracks_dev, tfade, stream);
      if (rc != PVK_OK) return rc;
    }
    int64_t gsz = (ntracks * 32 + 255) / 256;
    if (gsz > 148 * 16) gsz = 148 * 16;
    if (p.fcurve != nullptr)
      PVK_LAUNCH(resynth_tracks_kernel<true>, dim3((unsigned)gsz), dim3(256), 0, stream, p, ntracks, ntracks_dev, mask, tfade);
    else
      PVK_LAUNCH(resynth_tracks_kernel<false>, dim3((unsigned)gsz), dim3(256), 0, stream, p, ntracks, ntracks_dev, mask, tfade);
    PVK_CHECK_LAUNCH("pvk_resynth(tracks)");
  }
  // thread layout of the render kernel: RS samples per thread, nchp chunk threads per item
  // group, G item groups
  const int RS = hop >= 512 ? 16 : 8;
  const int nch = (hop + RS - 1) / RS;
  const int bd = nch >= 32 ? 128 : 64;                       // hops > bd*RS are rendered in windows
  p.nchp = nch < bd ? nch : bd;
  p.G = bd / p.nchp;
  if (p.G > npks) p.G = npks;
  if (hop % 128 == 0) {
    // tile kernels: bodies are built inside the render kernel, one launch over the whole block range
    p.chunk0 = block0;
    if (hop % 512 == 0) return launch_resynth_tile<16>(p, nblocks, stream);   // one warp per 512-sample tile
    if (hop % 256 == 0) return launch_resynth_tile<8>(p, nblocks, stream);
    return launch_resynth_tile<4>(p, nblocks, stream);                        // 128-sample tiles (16 kHz clip batches)
  }
  for (int64_t c0 = block0; c0 < block0 + nblocks; c0 += cb) {
    const int64_t n = (c0 + cb <= block0 + nblocks) ? cb : block0 + nblocks - c0;
    p.chunk0 = c0;
    p.block0 = c0;
    p.out = out + (c0 - block0) * (int64_t)hop;
    const dim3 pgrid((unsigned)((n + 3) / 4));
    if (p.fcurve != nullptr)
      PVK_LAUNCH((resynth_prepare_kernel<true, true>), pgrid, dim3(128), 0, stream, p, n, gitems, gcount);
    else if (p.free_phase)
      PVK_LAUNCH((resynth_prepare_kernel<true, false>), pgrid, dim3(128), 0, stream, p, n, gitems, gcount);
    else
      PVK_LAUNCH((resynth_prepare_kernel<false, false>), pgrid, dim3(128), 0, stream, p, n, gitems, gcount);
    PVK_CHECK_LAUNCH("pvk_resynth(prepare)");
    const int rc = RS == 16 ? launch_resynth<16>(p, n, bd, stream) : launch_resynth<8>(p, n, bd, stream);
    if (rc != PVK_OK) return rc;
  }
  return PVK_OK;
}

extern "C" int pvk_resynth_ex(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                              const int32_t *ntracks_dev, const int32_t *tstart, const int32_t *tlen,
                              const int64_t *toff, const double *pf, const double *pmag, const double *prealph,
                              double sr, int hop, int nfft, int hop_an, double edge, int minframes, double *out,
                              int64_t nout, int64_t block0, int64_t nblocks, void *workspace,
                              int64_t workspace_bytes, int reuse_tracks, int phase_preserve, double fscale,
                              double *phase_ws, int64_t phase_ws_len, void *stream) {
  return resynth_run(true, tid, nframes, npks, ntracks, ntracks_dev, tstart, tlen, toff, pf, pmag, prealph, sr, hop,
                     nfft, hop_an, edge, minframes, out, nout, block0, nblocks, workspace, workspace_bytes,
                     reuse_tracks, phase_preserve, fscale, nullptr, 0, phase_ws, phase_ws_len, stream);
}

extern "C" int pvk_resynth_ex_curve(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                                    const int32_t *ntracks_dev, const int32_t *tstart, const int32_t *tlen,
                                    const int64_t *toff, const double *pf, const double *pmag, const double *prealph,
                                    double sr, int hop, int nfft, int hop_an, double edge, int minframes, double *out,
                                    int64_t nout, int64_t block0, int64_t nblocks, void *workspace,
                                    int64_t workspace_bytes, int reuse_tracks, int phase_preserve, double fscale,
                                    const double *fcurve, int64_t fcurve_len, double *phase_ws, int64_t phase_ws_len,
                                    void *stream) {
  PVK_REQUIRE_CURVE("pvk_resynth_ex_curve", nframes, phase_preserve);
  return resynth_run(true, tid, nframes, npks, ntracks, ntracks_dev, tstart, tlen, toff, pf, pmag, prealph, sr, hop,
                     nfft, hop_an, edge, minframes, out, nout, block0, nblocks, workspace, workspace_bytes,
                     reuse_tracks, phase_preserve, fscale, fcurve, fcurve_len, phase_ws, phase_ws_len, stream);
}

extern "C" int pvk_resynth_render(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                                  const int32_t *ntracks_dev, const int32_t *tstart, const int32_t *tlen,
                                  const int64_t *toff, const double *pf, const double *pmag, const double *prealph,
                                  double sr, int hop, int nfft, int hop_an, double edge, int minframes, double *out,
                                  int64_t nout, int64_t block0, int64_t nblocks, void *workspace,
                                  int64_t workspace_bytes, int reuse_tracks, int phase_preserve, double fscale,
                                  double *phase_ws, int64_t phase_ws_len, void *stream) {
  PVK_REQUIRE(!phase_preserve, "pvk_resynth_render: phase_preserve=1 has no scan to leave out (use pvk_resynth_ex)");
  return resynth_run(false, tid, nframes, npks, ntracks, ntracks_dev, tstart, tlen, toff, pf, pmag, prealph, sr, hop,
                     nfft, hop_an, edge, minframes, out, nout, block0, nblocks, workspace, workspace_bytes,
                     reuse_tracks, phase_preserve, fscale, nullptr, 0, phase_ws, phase_ws_len, stream);
}

extern "C" int pvk_resynth_render_curve(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                                        const int32_t *ntracks_dev, const int32_t *tstart, const int32_t *tlen,
                                        const int64_t *toff, const double *pf, const double *pmag,
                                        const double *prealph, double sr, int hop, int nfft, int hop_an, double edge,
                                        int minframes, double *out, int64_t nout, int64_t block0, int64_t nblocks,
                                        void *workspace, int64_t workspace_bytes, int reuse_tracks, int phase_preserve,
                                        double fscale, const double *fcurve, int64_t fcurve_len, double *phase_ws,
                                        int64_t phase_ws_len, void *stream) {
  PVK_REQUIRE_CURVE("pvk_resynth_render_curve", nframes, phase_preserve);
  PVK_REQUIRE(!phase_preserve,
              "pvk_resynth_render_curve: phase_preserve=1 has no scan to leave out (use pvk_resynth_ex)");
  return resynth_run(false, tid, nframes, npks, ntracks, ntracks_dev, tstart, tlen, toff, pf, pmag, prealph, sr, hop,
                     nfft, hop_an, edge, minframes, out, nout, block0, nblocks, workspace, workspace_bytes,
                     reuse_tracks, phase_preserve, fscale, fcurve, fcurve_len, phase_ws, phase_ws_len, stream);
}

// ------------------------------------------------------------------ integrated phase across segments
// A rank of a segment-sharded run (dist.py) scans the partials of its window rows [w0, w1) only, so a
// partial alive at w0 starts there with the wrong phase, and its first Af + 1 advances read frames
// clamped at the cut.  From the hand-over row h = w0 + max(Af + 2, minframes) = j0 - dE on, the local
// advances are the true ones: P_local(r) - P_local(h) is exact for every r in [h, j1 + Lf - Af - 1)
// (fixed point, so the difference of two scanned values is the exact sum of the advances between them).
// Each rank records, for every column of the NEXT rank's hand-over row, either that difference and the
// partial's column in its own hand-over row or, for a partial born after its own hand-over row, the
// absolute P.  Composing the records of the ranks before g column by column gives the true P at row
// h(g); the partials alive there are shifted by seed - P_local(h(g)).  A rank whose window starts at
// frame 0 cuts nothing and records absolute values only, which ends every chain.
namespace pvk {

// record of column k of local row h_hi: rec[k] = column of the same partial in row h_lo (-1: absolute
// value, -2: no partial), rec[K + k] = P(h_hi) - P(h_lo) or P(h_hi), mod PHASE_ONE
__global__ void __launch_bounds__(128) handover_record_kernel(RParams p, int64_t ntracks, int64_t h_lo, int64_t h_hi,
                                                              int64_t *__restrict__ rec) {
  const int K = p.K;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < K; k += gridDim.x * blockDim.x) {
    int64_t col = -2;
    phase_t val = 0;
    const int v = h_hi >= 0 ? p.tid[h_hi * K + k] : -1;
    if (v >= 0 && v < ntracks) {
      const int64_t s = p.tstart[v], o = p.toff[v];
      if (o + (h_hi - s) < p.phcap) {
        val = p.phase[o + (h_hi - s)] & PHASE_MASK;
        col = -1;
        if (h_lo >= s) {                                           // alive at h_lo: relative to it
          for (int c = 0; c < K; ++c)
            if (p.tid[h_lo * K + c] == v) { col = c; break; }
          val = (val - p.phase[o + (h_lo - s)]) & PHASE_MASK;
        }
      }
    }
    rec[k] = col;
    rec[K + k] = (int64_t)val;
  }
}

// seed of column k of row h_lo from the records of ranks [0, rank) (recs [world][2K]), walked back from
// rank - 1 until an absolute value; delta[k] = seed - P_local(h_lo), dv[k] = the partial (-1: none)
__global__ void __launch_bounds__(128) handover_seed_kernel(RParams p, int64_t ntracks, const int64_t *__restrict__ recs,
                                                            int rank, int64_t h_lo, int64_t *__restrict__ delta,
                                                            int32_t *__restrict__ dv) {
  const int K = p.K;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < K; k += gridDim.x * blockDim.x) {
    const int v = p.tid[h_lo * K + k];
    int vv = -1;
    phase_t d = 0;
    if (v >= 0 && v < ntracks && p.toff[v] + (h_lo - p.tstart[v]) < p.phcap) {
      phase_t acc = 0;
      int c = k;
      for (int g = rank - 1; g >= 0; --g) {
        const int64_t col = recs[(int64_t)g * 2 * K + c];
        if (col < -1 || col >= K) break;                           // no partial there: records inconsistent
        acc = (acc + (phase_t)recs[(int64_t)g * 2 * K + K + c]) & PHASE_MASK;
        if (col == -1) {
          vv = v;
          d = (acc - p.phase[p.toff[v] + (h_lo - p.tstart[v])]) & PHASE_MASK;
          break;
        }
        c = (int)col;
      }
    }
    delta[k] = (int64_t)d;
    dv[k] = vv;
  }
}

// every point from row h_lo on of the partials alive at h_lo gets its column's delta added.  Points
// before h_lo keep a wrong P: nothing of an own block reads them (bodies start at j0 > h_lo, a tail reads
// the P of its partial's last row, and partials ending before h_lo = j0 - dE have no tail in an own block).
__global__ void __launch_bounds__(256) handover_fixup_kernel(RParams p, int64_t h_lo, const int64_t *__restrict__ delta,
                                                             const int32_t *__restrict__ dv, int nx) {
  const int k = blockIdx.x / nx, x = blockIdx.x % nx;
  const int v = dv[k];
  if (v < 0) return;
  const phase_t d = (phase_t)delta[k];
  const int64_t o = p.toff[v];
  int64_t n = p.tlen[v];
  if (o + n > p.phcap) n = p.phcap - o;
  for (int64_t i = (h_lo - p.tstart[v]) + (int64_t)x * blockDim.x + threadIdx.x; i < n; i += (int64_t)nx * blockDim.x)
    p.phase[o + i] = (p.phase[o + i] + d) & PHASE_MASK;
}

// global Nyquist flags: flags[gid[i]] = 1 for every point with fscale * f >= sr / 2 (the scan's test;
// CURVE: the ratio of the point's row i / K, fcurve[i / K], in place of fscale)
template <bool CURVE>
__global__ void __launch_bounds__(256) nyquist_scatter_kernel(const double *__restrict__ f, const int32_t *__restrict__ gid,
                                                              int64_t n, double sr, double fscale, uint8_t *flags,
                                                              int64_t nflags, const double *__restrict__ fcurve, int K) {
  const double nyq = 0.5 * sr;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int g = gid[i];
    const double r = CURVE ? fcurve[i / K] : fscale;
    if (g >= 0 && g < nflags && r * f[i] >= nyq && flags[g] == 0) flags[g] = 1;
  }
}

// one warp per local partial: its global id from the row of its first point, its flag into tfade[v].pad0
__global__ void __launch_bounds__(256) nyquist_import_kernel(RParams p, int64_t ntracks, const int32_t *__restrict__ table,
                                                             int64_t row0, const uint8_t *__restrict__ flags,
                                                             int64_t nflags, TrackFade *__restrict__ tfade) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < ntracks; v += nw) {
    const int64_t s = p.tstart[v];
    int g = -1;
    if (s >= 0 && s < p.F) {
      for (int c0 = 0; c0 < p.K; c0 += 32) {
        const int c = c0 + lane;
        const bool hit = c < p.K && p.tid[s * p.K + c] == (int)v;
        const unsigned m = __ballot_sync(FULL, hit);
        if (m) { g = table[(row0 + s) * p.K + c0 + __ffs((int)m) - 1]; break; }
      }
    }
    if (lane == 0) tfade[v].pad0 = (g >= 0 && g < nflags && flags[g]) ? 1 : 0;
  }
}

}  // namespace pvk

static TrackFade *resynth_tfade(void *workspace, int64_t nframes, int npks) {
  const int64_t mwk = (npks + 31) / 32;
  return reinterpret_cast<TrackFade *>(reinterpret_cast<unsigned char *>(workspace) + align_up(nframes * 2 * mwk * 4, 256));
}

#define PVK_REQUIRE_WS(fn)                                                                                          \
  PVK_REQUIRE(workspace != nullptr && workspace_bytes >= resynth_fixed_ws(nframes, npks, ntracks) +                 \
                                                             align_up(resynth_row_ws(npks), 256) + 512,             \
              fn ": workspace too small (%lld bytes; pvk_resynth_workspace_bytes gives the size)",                 \
              (long long)workspace_bytes)

static int resynth_scan_run(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks, const int32_t *tstart,
                            const int32_t *tlen, const int64_t *toff, const double *pf, const double *prealph,
                            double sr, int hop, int nfft, int hop_an, double fscale, const double *fcurve,
                            int64_t fcurve_len, void *workspace, int64_t workspace_bytes, double *phase_ws, int64_t phase_ws_len,
                            int64_t h_lo, int64_t h_hi, int64_t *rec, int64_t rec_len, void *stream) {
  PVK_REQUIRE(isfinite(fscale) && fscale > 0.0, "pvk_resynth_scan: fscale=%g must be finite and > 0", fscale);
  PVK_REQUIRE(hop >= 1 && nfft >= 1 && hop_an >= 1, "pvk_resynth_scan: hop=%d nfft=%d hop_an=%d must be >= 1", hop,
              nfft, hop_an);
  PVK_REQUIRE(npks >= 1 && npks <= PVK_MAX_NPKS, "pvk_resynth_scan: npks=%d must be in [1, %d]", npks, PVK_MAX_NPKS);
  PVK_REQUIRE(sr > 0.0, "pvk_resynth_scan: sr must be positive");
  PVK_REQUIRE(nframes >= 0 && ntracks >= 0, "pvk_resynth_scan: negative sizes");
  PVK_REQUIRE(nframes == 0 || ntracks == 0 || (tid && tstart && tlen && toff && pf && prealph),
              "pvk_resynth_scan: NULL pointer argument");
  PVK_REQUIRE(h_lo < nframes && h_hi < nframes, "pvk_resynth_scan: hand-over rows %lld / %lld outside the %lld rows",
              (long long)h_lo, (long long)h_hi, (long long)nframes);
  PVK_REQUIRE(h_hi < 0 || h_lo <= h_hi, "pvk_resynth_scan: h_lo=%lld after h_hi=%lld", (long long)h_lo, (long long)h_hi);
  PVK_REQUIRE(rec == nullptr || rec_len >= 2 * (int64_t)npks, "pvk_resynth_scan: rec_len=%lld is short (2 * npks = %d)",
              (long long)rec_len, 2 * npks);
  const int64_t need = ntracks < nframes * (int64_t)npks ? ntracks : nframes * (int64_t)npks;
  PVK_REQUIRE(phase_ws != nullptr && phase_ws_len >= need,
              "pvk_resynth_scan: phase_ws_len=%lld is short (one double per packed point, at least %lld)",
              (long long)phase_ws_len, (long long)need);
  PVK_REQUIRE_WS("pvk_resynth_scan");
  RParams p;
  synth_params(p, sr, hop, nfft, hop_an, npks, fscale);
  p.tid = tid; p.tstart = tstart; p.tlen = tlen; p.toff = toff; p.pf = pf; p.prealph = prealph;
  p.F = nframes; p.ntcap = ntracks;
  p.phase = reinterpret_cast<unsigned long long *>(phase_ws);
  p.phcap = phase_ws_len;
  p.free_phase = 1;
  p.fcurve = fcurve;
  p.fcurve_len = fcurve_len;
  if (ntracks > 0 && nframes > 0) {
    const int rc = launch_phase_scan(p, ntracks, nullptr, resynth_tfade(workspace, nframes, npks), stream);
    if (rc != PVK_OK) return rc;
  }
  if (rec != nullptr) {
    PVK_LAUNCH(handover_record_kernel, dim3((unsigned)((npks + 127) / 128)), dim3(128), 0, stream, p,
               nframes > 0 ? ntracks : 0, h_lo, nframes > 0 ? h_hi : -1, rec);
    PVK_CHECK_LAUNCH("pvk_resynth_scan(record)");
  }
  return PVK_OK;
}

extern "C" int pvk_resynth_scan(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks, const int32_t *tstart,
                                const int32_t *tlen, const int64_t *toff, const double *pf, const double *prealph,
                                double sr, int hop, int nfft, int hop_an, double fscale, void *workspace,
                                int64_t workspace_bytes, double *phase_ws, int64_t phase_ws_len, int64_t h_lo,
                                int64_t h_hi, int64_t *rec, int64_t rec_len, void *stream) {
  return resynth_scan_run(tid, nframes, npks, ntracks, tstart, tlen, toff, pf, prealph, sr, hop, nfft, hop_an, fscale,
                          nullptr, 0, workspace, workspace_bytes, phase_ws, phase_ws_len, h_lo, h_hi, rec, rec_len, stream);
}

extern "C" int pvk_resynth_scan_curve(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                                      const int32_t *tstart, const int32_t *tlen, const int64_t *toff, const double *pf,
                                      const double *prealph, double sr, int hop, int nfft, int hop_an, double fscale,
                                      const double *fcurve, int64_t fcurve_len, void *workspace,
                                      int64_t workspace_bytes, double *phase_ws, int64_t phase_ws_len, int64_t h_lo,
                                      int64_t h_hi, int64_t *rec, int64_t rec_len, void *stream) {
  PVK_REQUIRE_CURVE("pvk_resynth_scan_curve", nframes, 0);
  return resynth_scan_run(tid, nframes, npks, ntracks, tstart, tlen, toff, pf, prealph, sr, hop, nfft, hop_an, fscale,
                          fcurve, fcurve_len, workspace, workspace_bytes, phase_ws, phase_ws_len, h_lo, h_hi, rec, rec_len, stream);
}

extern "C" int pvk_resynth_handover(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                                    const int32_t *tstart, const int32_t *tlen, const int64_t *toff, double *phase_ws,
                                    int64_t phase_ws_len, const int64_t *recs, int64_t recs_len, int world, int rank,
                                    int64_t h_lo, void *workspace, int64_t workspace_bytes, void *stream) {
  PVK_REQUIRE(npks >= 1 && npks <= PVK_MAX_NPKS, "pvk_resynth_handover: npks=%d must be in [1, %d]", npks,
              PVK_MAX_NPKS);
  PVK_REQUIRE(nframes >= 0 && ntracks >= 0, "pvk_resynth_handover: negative sizes");
  PVK_REQUIRE(world >= 1 && rank >= 0 && rank < world, "pvk_resynth_handover: rank=%d outside world=%d", rank, world);
  PVK_REQUIRE(h_lo < nframes, "pvk_resynth_handover: h_lo=%lld outside the %lld rows", (long long)h_lo,
              (long long)nframes);
  PVK_REQUIRE(recs != nullptr && recs_len >= (int64_t)world * 2 * npks,
              "pvk_resynth_handover: recs_len=%lld is short (world * 2 * npks = %lld)", (long long)recs_len,
              (long long)world * 2 * npks);
  PVK_REQUIRE(nframes == 0 || ntracks == 0 || (tid && tstart && tlen && toff && phase_ws),
              "pvk_resynth_handover: NULL pointer argument");
  PVK_REQUIRE(phase_ws_len >= 0, "pvk_resynth_handover: negative phase_ws_len");
  PVK_REQUIRE_WS("pvk_resynth_handover");
  if (h_lo < 0 || rank == 0 || nframes == 0 || ntracks == 0) return PVK_OK;     // nothing cut: the scan is exact
  RParams p;
  p.tid = tid; p.tstart = tstart; p.tlen = tlen; p.toff = toff;
  p.F = nframes; p.K = npks; p.ntcap = ntracks;
  p.phase = reinterpret_cast<unsigned long long *>(phase_ws);
  p.phcap = phase_ws_len;
  // delta / dv live in the chunk area of the workspace (the render stage rewrites it)
  unsigned char *scratch = reinterpret_cast<unsigned char *>(workspace) + resynth_fixed_ws(nframes, npks, ntracks);
  int64_t *delta = reinterpret_cast<int64_t *>(scratch);
  int32_t *dv = reinterpret_cast<int32_t *>(scratch + 8 * (int64_t)npks);
  PVK_LAUNCH(handover_seed_kernel, dim3((unsigned)((npks + 127) / 128)), dim3(128), 0, stream, p, ntracks, recs, rank,
             h_lo, delta, dv);
  PVK_CHECK_LAUNCH("pvk_resynth_handover(seed)");
  const int nx = 32;
  PVK_LAUNCH(handover_fixup_kernel, dim3((unsigned)(npks * nx)), dim3(256), 0, stream, p, h_lo, delta, dv, nx);
  PVK_CHECK_LAUNCH("pvk_resynth_handover(fix-up)");
  return PVK_OK;
}

static int nyquist_flags_run(const double *f, const int32_t *gid, int64_t n, double sr, double fscale,
                             const double *fcurve, int npks, uint8_t *flags, int64_t nflags, void *stream) {
  PVK_REQUIRE(isfinite(fscale) && fscale > 0.0, "pvk_nyquist_flags: fscale=%g must be finite and > 0", fscale);
  PVK_REQUIRE(sr > 0.0, "pvk_nyquist_flags: sr must be positive");
  PVK_REQUIRE(n >= 0 && nflags >= 0, "pvk_nyquist_flags: negative sizes");
  PVK_REQUIRE(n == 0 || (f && gid), "pvk_nyquist_flags: NULL pointer argument");
  PVK_REQUIRE(nflags == 0 || flags, "pvk_nyquist_flags: flags is NULL");
  if (n == 0 || nflags == 0) return PVK_OK;
  int64_t g = (n + 255) / 256;
  if (g > 148 * 8) g = 148 * 8;
  if (fcurve != nullptr)
    PVK_LAUNCH(nyquist_scatter_kernel<true>, dim3((unsigned)g), dim3(256), 0, stream, f, gid, n, sr, fscale, flags, nflags,
               fcurve, npks);
  else
    PVK_LAUNCH(nyquist_scatter_kernel<false>, dim3((unsigned)g), dim3(256), 0, stream, f, gid, n, sr, fscale, flags,
               nflags, nullptr, 1);
  PVK_CHECK_LAUNCH("pvk_nyquist_flags");
  return PVK_OK;
}

extern "C" int pvk_nyquist_flags(const double *f, const int32_t *gid, int64_t n, double sr, double fscale,
                                 uint8_t *flags, int64_t nflags, void *stream) {
  return nyquist_flags_run(f, gid, n, sr, fscale, nullptr, 1, flags, nflags, stream);
}

extern "C" int pvk_nyquist_flags_curve(const double *f, const int32_t *gid, int64_t n, double sr, double fscale,
                                       const double *fcurve, int64_t fcurve_len, int npks, uint8_t *flags,
                                       int64_t nflags, void *stream) {
  PVK_REQUIRE(npks >= 1 && npks <= PVK_MAX_NPKS, "pvk_nyquist_flags_curve: npks=%d must be in [1, %d]", npks,
              PVK_MAX_NPKS);
  PVK_REQUIRE(n >= 0 && n % npks == 0, "pvk_nyquist_flags_curve: n=%lld is not a whole number of rows of %d",
              (long long)n, npks);
  PVK_REQUIRE_CURVE("pvk_nyquist_flags_curve", n / npks, 0);
  return nyquist_flags_run(f, gid, n, sr, fscale, fcurve, npks, flags, nflags, stream);
}

extern "C" int pvk_resynth_import_flags(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                                        const int32_t *tstart, const int32_t *table, int64_t table_rows, int64_t row0,
                                        const uint8_t *flags, int64_t nflags, void *workspace, int64_t workspace_bytes,
                                        void *stream) {
  PVK_REQUIRE(npks >= 1 && npks <= PVK_MAX_NPKS, "pvk_resynth_import_flags: npks=%d must be in [1, %d]", npks,
              PVK_MAX_NPKS);
  PVK_REQUIRE(nframes >= 0 && ntracks >= 0 && nflags >= 0 && table_rows >= 0, "pvk_resynth_import_flags: negative sizes");
  PVK_REQUIRE(row0 >= 0 && row0 + nframes <= table_rows,
              "pvk_resynth_import_flags: rows [%lld, %lld) outside the table's %lld rows", (long long)row0,
              (long long)(row0 + nframes), (long long)table_rows);
  PVK_REQUIRE(nframes == 0 || ntracks == 0 || (tid && tstart && table), "pvk_resynth_import_flags: NULL pointer argument");
  PVK_REQUIRE(nflags == 0 || flags, "pvk_resynth_import_flags: flags is NULL");
  PVK_REQUIRE_WS("pvk_resynth_import_flags");
  if (nframes == 0 || ntracks == 0) return PVK_OK;
  RParams p;
  p.tid = tid; p.tstart = tstart;
  p.F = nframes; p.K = npks;
  int64_t g = (ntracks * 32 + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  PVK_LAUNCH(nyquist_import_kernel, dim3((unsigned)g), dim3(256), 0, stream, p, ntracks, table, row0, flags, nflags,
             resynth_tfade(workspace, nframes, npks));
  PVK_CHECK_LAUNCH("pvk_resynth_import_flags");
  return PVK_OK;
}
