// pvk_analyze.cu -- fused phase-vocoder analysis kernel for sm_100a.
//
// One CTA walks a run of consecutive STFT frames of one signal (analyze_kernel: one frame at a
// time; analyze_warp_kernel, nfft 1024 / 2048: one warp per frame, AW frames at a time, same
// results bit for bit).  Per frame, without ever
// leaving shared memory / registers:
//   1. framing + windowing: the hop-strided frame is read straight from the signal with
//      coalesced 64-bit loads (re-reads of the nfft-hop overlap hit L1/L2, HBM sees each
//      sample about once) and multiplied by win/wfact            (PVAnalysis.py:155-157)
//   2. real FFT of nfft points as a complex Stockham FFT of M = nfft/2 points (radix-16/8/4
//      register butterflies, padded shared-memory exchanges) plus an in-place untangle step
//      that yields bins 0..M-1 = fx[:nfft/2]                     (PVAnalysis.py:157,169)
//   3. peak picking on |fx| with PeakFinder's exact semantics: local maxima, strict
//      threshold, top-npks by (value desc, bin asc) through an exact radix select on the
//      fp32 bit pattern, ascending-bin order, +-5-bin salience filter
//                                                (PeakFinder.py:57-70,155-194,113-134)
//   4. per-peak epilogue in fp64 with the reference's operation order: phase, phase
//      difference against the previous frame's spectrum (kept in the other half of a
//      shared-memory double buffer), dphase2freq, 3-bin magnitude, realph, freq>0 filter
//                                                (PVAnalysis.py:133-147,187-207)
//   5. zero padded float64 rows in the reference's layout        (PVAnalysis.py:226-245)
// Not a dense contraction: no tensor cores.  fp32 FFT, fp64 only per peak.
#include "pvk_common.cuh"

namespace pvk {

#define PADC(i) ((i) + ((i) >> 4))
// |fx| lives in shared memory with 4 pad words per 16 bins: a thread reads its contiguous run of
// bins with 128-bit loads, conflict free
#define FA(i) ((i) + (((i) >> 4) << 2))

struct AParams {
  const float *x;
  int64_t clip_stride;
  const float *win;
  const float2 *tables;
  const double *fbin;
  const double *wfbin;
  int hop, npks;
  double pkthresh, dt, fstep;
  int64_t frame0, nframes;
  int64_t out_rows;              // rows per clip of the output tables (>= nframes; the rest are the caller's guard rows)
  int prev_zero, run;
  int64_t nruns;
  double *f, *mag, *ph, *realph, *binno;
  int32_t *npk;
  double *totalmag;
  float2 *spec_out;
  double *fine_pos, *fine_val;   // optional PeakFinder.refine outputs (PeakFinder.py:331-372)
};

template <int LOGM> struct Plan {
  static constexpr int M = 1 << LOGM;
  // (at most 512 threads = 16 warps per CTA: the per-warp reduction slots of Smem are sized for that)
  static constexpr int LOGT = LOGM <= 8 ? 5 : (LOGM <= 10 ? 6 : LOGM - 4);
  static constexpr int T = 1 << LOGT;
  static constexpr int LP0 = LOGM - LOGT;
  static constexpr int LP = LP0 < 2 ? 2 : (LP0 > 4 ? 4 : LP0);
  static constexpr int NPASS = (LOGM + LP - 1) / LP;
  __host__ __device__ static constexpr int lr(int q) { return q < NPASS - 1 ? LP : LOGM - LP * (NPASS - 1); }
  __host__ __device__ static constexpr int lp(int q) { return q * LP; }
  __host__ __device__ static constexpr int tw_off(int q) {
    int o = 0;
    for (int i = 1; i < q; ++i) o += ((1 << lr(i)) - 1) << lp(i);
    return o;
  }
  static constexpr int TW_TOTAL = tw_off(NPASS);
  static constexpr int MP = M + (M >> 4) + 1;
  static constexpr int NW = T / 32;
};

// ------------------------------------------------------------------ small DFTs
template <int LR> __host__ __device__ constexpr int brev(int s) {
  int r = 0;
  for (int b = 0; b < LR; ++b) r |= ((s >> b) & 1) << (LR - 1 - b);
  return r;
}

// d * W_16^e, W_16 = exp(-2*pi*i/16), e in [0,8)
__device__ __forceinline__ float2 mul_w16(float2 d, int e) {
  const float C8 = 0.70710678118654752440f, C1 = 0.92387953251128675613f, S1 = 0.38268343236508977173f;
  switch (e) {
    case 0: return d;
    case 4: return make_float2(d.y, -d.x);
    case 2: return make_float2((d.x + d.y) * C8, (d.y - d.x) * C8);
    case 6: return make_float2((d.y - d.x) * C8, -(d.x + d.y) * C8);
    case 1: return make_float2(d.x * C1 + d.y * S1, d.y * C1 - d.x * S1);
    case 3: return make_float2(d.x * S1 + d.y * C1, d.y * S1 - d.x * C1);
    case 5: return make_float2(d.y * C1 - d.x * S1, -d.y * S1 - d.x * C1);
    default: return make_float2(d.y * S1 - d.x * C1, -d.y * C1 - d.x * S1);  // e == 7
  }
}

// in-register DFT of R = 2^LR points, radix-2 DIF stages; result V[s] ends up in u[brev(s)]
template <int LR> __device__ __forceinline__ void dft_dif(float2 *u) {
  constexpr int R = 1 << LR;
#pragma unroll
  for (int h = R / 2; h >= 1; h >>= 1) {
#pragma unroll
    for (int g = 0; g < R; g += 2 * h) {
#pragma unroll
      for (int j = 0; j < h; ++j) {
        float2 a = u[g + j], b = u[g + j + h];
        u[g + j] = make_float2(a.x + b.x, a.y + b.y);
        float2 d = make_float2(a.x - b.x, a.y - b.y);
        u[g + j + h] = mul_w16(d, j * (8 / h));
      }
    }
  }
}

__device__ __forceinline__ float2 cmul(float2 a, float2 w) {
  return make_float2(a.x * w.x - a.y * w.y, a.x * w.y + a.y * w.x);
}

// ------------------------------------------------------------------ FFT passes
template <int LOGM, int Q> struct Pass {
  using P = Plan<LOGM>;
  static constexpr int M = P::M, T = P::T;
  static constexpr int LR = P::lr(Q), R = 1 << LR, LPQ = P::lp(Q), PP = 1 << LPQ;
  static constexpr int NBF = M >> LR, NB = (NBF + T - 1) / T;
  static constexpr int OFF = P::tw_off(Q);

  static __device__ __forceinline__ void run(const float2 *__restrict__ twp, float2 *buf) {
    const int tid = threadIdx.x;
    float2 u[NB][R];
    // twiddles first: their loads overlap the shared-memory reads and the barrier
    float2 tw[NB * (R - 1) > 0 ? NB * (R - 1) : 1];
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      const int i = tid + b * T;
      if (NBF >= T || i < NBF) {
        const int k = i & (PP - 1);
#pragma unroll
        for (int r = 1; r < R; ++r) tw[b * (R - 1) + r - 1] = __ldg(twp + OFF + (r - 1) * PP + k);
      }
    }
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      const int i = tid + b * T;
      if (NBF >= T || i < NBF) {
#pragma unroll
        for (int r = 0; r < R; ++r) u[b][r] = buf[PADC(i + r * NBF)];
      }
    }
    __syncthreads();
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      const int i = tid + b * T;
      if (NBF >= T || i < NBF) {
        const int k = i & (PP - 1);
        const int j = ((i - k) << LR) + k;
#pragma unroll
        for (int r = 1; r < R; ++r) u[b][r] = cmul(u[b][r], tw[b * (R - 1) + r - 1]);
        dft_dif<LR>(u[b]);
#pragma unroll
        for (int s = 0; s < R; ++s) buf[PADC(j + s * PP)] = u[b][brev<LR>(s)];
      }
    }
    __syncthreads();
    if constexpr (Q + 1 < P::NPASS) Pass<LOGM, Q + 1>::run(twp, buf);
  }
};

// Two consecutive signal samples: one 64-bit load when p is 8-byte aligned (al8)
__device__ __forceinline__ float2 ldg_stream2(const float *p, bool al8) {
  if (al8) return __ldg(reinterpret_cast<const float2 *>(p));
  return make_float2(__ldg(p), __ldg(p + 1));
}

// samples of one frame -> registers: thread `tid` gets the packed points z[m] = (x[2m], x[2m+1]),
// m = tid + r * NBF, that its first butterfly needs (raw samples, the window is applied by
// fft_frame_regs).  Issued one phase ahead of the FFT that consumes them (analyze_kernel).
template <int LOGM>
__device__ __forceinline__ void frame_load(const float *__restrict__ xf, float2 *u) {
  using P = Plan<LOGM>;
  constexpr int M = P::M, T = P::T;
  constexpr int LR = P::lr(0), R = 1 << LR;
  constexpr int NBF = M >> LR;
  static_assert(NBF <= T, "one first-pass butterfly per thread");
  const int i = threadIdx.x;
  const bool al8 = ((reinterpret_cast<uintptr_t>(xf) & 7) == 0);
  if (NBF >= T || i < NBF) {
#pragma unroll
    for (int r = 0; r < R; ++r) u[r] = ldg_stream2(xf + 2 * (i + r * NBF), al8);
  }
}

// complex FFT of the windowed frame held in u[] (frame_load), packed z[m] = (x[2m], x[2m+1]);
// natural order in buf
template <int LOGM>
__device__ __forceinline__ void fft_frame_regs(float2 *u, const float *__restrict__ win,
                                               const float2 *__restrict__ twp, float2 *buf) {
  using P = Plan<LOGM>;
  constexpr int M = P::M, T = P::T;
  constexpr int LR = P::lr(0), R = 1 << LR;
  constexpr int NBF = M >> LR;
  const int i = threadIdx.x;
  if (NBF >= T || i < NBF) {
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const float2 wv = __ldg(reinterpret_cast<const float2 *>(win) + i + r * NBF);
      u[r] = make_float2(u[r].x * wv.x, u[r].y * wv.y);
    }
    dft_dif<LR>(u);
#pragma unroll
    for (int s = 0; s < R; ++s) buf[PADC(i * R + s)] = u[brev<LR>(s)];
  }
  __syncthreads();
  if constexpr (P::NPASS > 1) Pass<LOGM, 1>::run(twp, buf);
}

template <int LOGM>
__device__ __forceinline__ void fft_frame(const float *__restrict__ xf, const float *__restrict__ win,
                                          const float2 *__restrict__ twp, float2 *buf) {
  float2 u[1 << Plan<LOGM>::lr(0)];
  frame_load<LOGM>(xf, u);
  fft_frame_regs<LOGM>(u, win, twp, buf);
}

// ------------------------------------------------------------------ per-peak epilogue
struct PeakVals { double f, mag, ph, realph; };

// np.angle(fx[k]) and dphase2freq(np.angle((fx/oldfft)[k]), k): PVAnalysis.py:188-191 +
// :133-147, in fp64 and in the reference's operation order (explicit _rn intrinsics: no FMA
// contraction where rounding decides ties).  bf = freq, bdf = fbin[k] - freq.
__device__ __forceinline__ void peak_phase_freq_exact(float2 c, float2 p, int k,
                                                      const double *__restrict__ fbin,
                                                      const double *__restrict__ wfbin, double dt, double inv,
                                                      double step, double &thisph, double &bf, double &bdf) {
  const double re = c.x, im = c.y, ore = p.x, oim = p.y;
  thisph = atan2(im, re);                                    // np.angle(fx[nbin]) :188
  // frat = fx / oldfft (:171): numpy's complex128 division (Smith), incl. the x/0 case.  Only the
  // ANGLE of the quotient is used (:190), so the common positive factor 1/|denominator| of Smith's
  // formula is dropped (its sign is kept): one fp64 division less, angle equal to ~1 ulp.
  double qr, qi;
  const double ar = fabs(ore), ai = fabs(oim);
  if (ar >= ai) {
    if (ar == 0.0 && ai == 0.0) {
      qr = re / ar; qi = im / ar;                            // (+-inf | nan, +-inf | nan)
    } else {
      const double rat = oim / ore, den = ore + oim * rat;
      qr = re + im * rat; qi = im - re * rat;
      if (den < 0.0) { qr = -qr; qi = -qi; }
    }
  } else {
    const double rat = ore / oim, den = oim + ore * rat;
    qr = re * rat + im; qi = im * rat - re;
    if (den < 0.0) { qr = -qr; qi = -qi; }
  }
  const double dph = atan2(qi, qr);                          // np.angle(frat[nbin]) :190
  const double PI2 = 6.283185307179586;
  const double fb = __ldg(fbin + k);
  const double base = __dadd_rn(dph, __ldg(wfbin + k));      // :140
  // :141-147: freq_m = (base + 2 pi {-1,0,1}) / dt / 2 pi, pick the first minimum of |fbin - freq_m|.
  // The candidates are one frame rate (1/dt) apart, so the winner is decided on a
  // multiply-by-reciprocal estimate unless two of them are within 1e-9 (relative) of a tie; the
  // reference's two correctly rounded divisions are then made for the winner only.
  // (inv = 1 / (2 pi dt), step = 1 / dt: computed once per kernel)
  const double e1 = fb - base * inv;                         // df estimate of m = 1; m = 0 / 2 are +- step away
  const double a0 = fabs(e1 + step), a1 = fabs(e1), a2 = fabs(e1 - step);
  int best = a0 <= a1 ? (a0 <= a2 ? 0 : 2) : (a1 <= a2 ? 1 : 2);
  const double lo = fmin(a0, fmin(a1, a2));
  const double second = best == 0 ? fmin(a1, a2) : (best == 1 ? fmin(a0, a2) : fmin(a0, a1));
  const bool clear = (second - lo) > 1e-9 * step;            // false for NaN as well
  if (clear) {
    const double dphw = __dadd_rn(base, best == 0 ? -PI2 : (best == 1 ? 0.0 : PI2));
    bf = __ddiv_rn(__ddiv_rn(dphw, dt), PI2);                // :142
    bdf = __dsub_rn(fb, bf);                                 // :144
  } else {
    double ba = 0.0;
    bf = 0.0; bdf = 0.0;
#pragma unroll
    for (int m = 0; m < 3; ++m) {
      const double dphw = __dadd_rn(base, m == 0 ? -PI2 : (m == 1 ? 0.0 : PI2));
      const double fq = __ddiv_rn(__ddiv_rn(dphw, dt), PI2); // :142
      const double df = __dsub_rn(fb, fq);                   // :144
      const double a = fabs(df);
      if (m == 0 || a < ba) { bf = fq; bdf = df; ba = a; }   // np.argmin: first minimum, nan sticks
    }
  }
}

__device__ __forceinline__ void peak_phase_freq(int k, const float2 *cur, const float2 *prev,
                                                const double *__restrict__ fbin,
                                                const double *__restrict__ wfbin, double dt, double inv,
                                                double step, double &thisph, double &bf, double &bdf) {
  peak_phase_freq_exact(cur[PADC(k)], prev[PADC(k)], k, fbin, wfbin, dt, inv, step, thisph, bf, bdf);
}

// out-of-line copy of the exact path for analyze_kernel's rare cases (keeps its registers off the hot path)
__device__ __noinline__ void peak_phase_freq_slow(float2 c, float2 p, int k, const double *__restrict__ fbin,
                                                  const double *__restrict__ wfbin, double dt, double inv,
                                                  double step, double *out3) {
  double thisph, bf, bdf;
  peak_phase_freq_exact(c, p, k, fbin, wfbin, dt, inv, step, thisph, bf, bdf);
  out3[0] = thisph; out3[1] = bf; out3[2] = bdf;
}

// The same three results on the fp32 pipes: the spectrum is an fp32 FFT (relative error ~1e-7), so
// the two angles are taken with atan2f (<= 2 ulp, ~3e-7 rad; north-star tolerance 1e-4 rad) -- the
// angle of the quotient fx/oldfft as the angle of fx * conj(oldfft).  Everything that DECIDES
// something still follows the reference exactly: whenever the unwrap candidates are within
// 1e-5 of a tie (fp32 moves a candidate by ~5e-8 of their spacing), the frequency is within 1e-4
// frame rates of zero (the freq > 0 filter, :193), or the previous bin is zero / the product under-
// or overflows (numpy's x/0 semantics), the exact fp64 path above is taken instead.
constexpr double RINT_MAGIC_A = 6755399441055744.0;             // 1.5 * 2^52: (x + M) - M == rint(x)
__device__ __forceinline__ void peak_phase_freq_fast(int k, const float2 *cur, const float2 *prev,
                                                     const double *__restrict__ fbin,
                                                     const double *__restrict__ wfbin, double dt, double inv,
                                                     double step, double &thisph, double &bf, double &bdf) {
  const float2 c = cur[PADC(k)], p = prev[PADC(k)];
  const float qr = fmaf(c.x, p.x, c.y * p.y), qi = fmaf(c.y, p.x, -(c.x * p.y));
  const float qn = fabsf(qr) + fabsf(qi);
  bool ok = qn > 1e-30f && qn < 1e30f;                        // false for NaN / inf / 0 as well
  const double PI2 = 6.283185307179586;
  const double fb = __ldg(fbin + k);
  if (ok) {
    const double base = (double)atan2f(qi, qr) + __ldg(wfbin + k);   // :140
    // :141-147 in closed form: the candidates base + 2 pi {-1, 0, 1} are one frame rate (1/dt) apart
    // in frequency and the one nearest the bin centre wins, i.e. base + 2 pi clamp(rint(t), -1, 1)
    // with t = df of the middle candidate in frame rates; two candidates tie at |t| = 0.5, where
    // np.argmin takes the first (left to the exact path)
    const double t = (fb - base * inv) * dt;
    const double mr = fmax(-1.0, fmin(1.0, (t + RINT_MAGIC_A) - RINT_MAGIC_A));
    bf = fma(mr, PI2, base) * inv;                            // :142
    bdf = fb - bf;                                            // :144
    ok = fabs(fabs(t) - 0.5) > 1e-5 && fabs(bf) > 1e-4 * step;
    thisph = (double)atan2f(c.y, c.x);                        // :188
  }
  if (!ok) {
    double o3[3];
    peak_phase_freq_slow(c, p, k, fbin, wfbin, dt, inv, step, o3);
    thisph = o3[0]; bf = o3[1]; bdf = o3[2];
  }
}

// |fx[k]|^2 in fp32 without FMA contraction (bit-identical to numpy float32 re*re + im*im)
__device__ __forceinline__ float bin_power(float2 c) { return __fadd_rn(__fmul_rn(c.x, c.x), __fmul_rn(c.y, c.y)); }

// Where the per-bin powers come from: analyze_kernel stores them (famp), analyze_warp_kernel
// recomputes them from the untangled spectrum with bin_power -- the same bits either way.
struct FampPow {
  const float *famp;
  __device__ __forceinline__ float operator()(int k) const { return famp[FA(k)]; }
};
struct SpecPow {
  const float2 *spec;
  __device__ __forceinline__ float operator()(int k) const { return bin_power(spec[PADC(k)]); }
};

// PVAnalysis.py:188-207 for the peak at bin k (1 <= k <= M-2)
template <class Pow>
__device__ __forceinline__ bool peak_epilogue(int k, int M, const float2 *cur, const float2 *prev,
                                              const Pow &famp, const double *__restrict__ fbin,
                                              const double *__restrict__ wfbin, double dt, double inv,
                                              double step, double pi_fstep, PeakVals &o) {
  double thisph, bf, bdf;
  peak_phase_freq_fast(k, cur, prev, fbin, wfbin, dt, inv, step, thisph, bf, bdf);
  // mag = sqrt(sum(famp[max(nbin-1,1) : min(nbin+1,len)+1]**2)), left to right :197-199; famp holds
  // the fp32 powers |fx|^2, summed and rooted in fp32 (relative error ~2e-7, tolerance 1e-4)
  float s = famp(k);
  if (k - 1 >= 1) s = famp(k - 1) + s;
  if (k + 1 <= M - 1) s = s + famp(k + 1);
  o.f = bf;
  o.mag = (double)sqrtf(s);
  o.ph = thisph;
  o.realph = fma(bdf, pi_fstep, thisph);                     // :207 ph + pi*df/fstep
  return bf > 0.0;                                           // :193 (drops nan too)
}

// PeakFinder.refine (PeakFinder.py:331-372, fun=None, x = arange): parabola through
// famp[k-1], famp[k], famp[k+1] (famp = sqrt of the stored power) -> fine position and value;
// a bin that is not a local maximum keeps (k, famp[k]).  1 <= k <= M-2.
template <class Pow> __device__ __forceinline__ void refine_peak(int k, const Pow &famp, double &fpos, double &fval) {
  const double s0 = sqrt((double)famp(k - 1)), s1 = sqrt((double)famp(k)), s2 = sqrt((double)famp(k + 1));
  if (s1 > s0 && s1 >= s2) {                                 // :354
    const double c = s1;
    const double b = __ddiv_rn(__dsub_rn(s2, s0), 2.0);
    const double a = __dsub_rn(__ddiv_rn(__dadd_rn(s2, s0), 2.0), c);
    const double lpos = __ddiv_rn(__ddiv_rn(-b, 2.0), a);    // - b/2/a
    fpos = __dadd_rn((double)k, lpos);
    fval = __dadd_rn(__dadd_rn(__dmul_rn(__dmul_rn(a, lpos), lpos), __dmul_rn(b, lpos)), c);   // :365
  } else {
    fpos = (double)k;
    fval = s1;
  }
}

// ------------------------------------------------------------------ the kernel
template <int LOGM> struct Smem {
  using P = Plan<LOGM>;
  static constexpr int OFF_BUF0 = 0;
  static constexpr int OFF_BUF1 = OFF_BUF0 + P::MP * 8;
  static constexpr int OFF_FAMP = OFF_BUF1 + P::MP * 8;
  static constexpr int OFF_HIST = OFF_FAMP + (P::M + P::M / 4 + 4) * 4;
  static constexpr int OFF_RED = (OFF_HIST + 3 * 128 * 4 + 7) / 8 * 8;   // doubles: one sum per warp (<= 16 warps)
  static constexpr int OFF_REDF = OFF_RED + 16 * 8;                  // floats: 16 min, 16 max
  static constexpr int OFF_REDU = OFF_REDF + 32 * 4;                 // uints: 16 cnt, 16 kmin, 16 kmax
  static constexpr int OFF_BC = OFF_REDU + 48 * 4;                   // 8 broadcast ints
  static constexpr int OFF_WS = OFF_BC + 8 * 4;                      // 2 x (2 x 16) warp sums
  static constexpr int OFF_CBIN = OFF_WS + 64 * 4;                   // candidate bins (uint16, compact)
  static constexpr int OFF_SELW = OFF_CBIN + P::M * 2;               // 2 x M/32 ballot words
  static constexpr int OFF_PK = OFF_SELW + 2 * (P::M / 32) * 4;      // 2 x npks uint16
  static int bytes(int npks) { return OFF_PK + 2 * ((npks + 7) / 8 * 8) * 2; }
};

// Ordered compaction of a list processed in rounds of blockDim threads: position of this
// thread's entry among the flagged ones (valid if flag), running total in `base`.
// wsum: 2 x NW ints, double buffered by round parity -> one barrier per round.
template <int NW>
__device__ __forceinline__ int round_pos(bool flag, int *wsum, int round, int &base) {
  const unsigned m = __ballot_sync(FULL, flag);
  int *ws = wsum + (round & 1) * NW;
  if (lane_id() == 0) ws[warp_id()] = __popc(m);
  __syncthreads();
  int wb = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < NW; ++w) { const int c = ws[w]; wb += (w < warp_id()) ? c : 0; tot += c; }
  const int pos = base + wb + __popc(m & lanemask_lt());
  base += tot;
  return pos;
}

template <int LOGM>
__global__ void __launch_bounds__(Plan<LOGM>::T, 512 / Plan<LOGM>::T) analyze_kernel(AParams prm) {
  using P = Plan<LOGM>;
  using S = Smem<LOGM>;
  constexpr int M = P::M, T = P::T, NW = P::NW, N = 2 * M;
  constexpr int CB = M / T;                                  // contiguous bins per thread in the candidate scan
  PVK_SMEM(smem);
  // the two spectrum buffers are addressed as smem + parity * stride (not through an array of
  // pointers): the compiler then keeps the accesses in the shared state space (LDS / STS instead of
  // generic LD / ST, and no pointer table on the local stack)
  constexpr int BUF_STRIDE = S::OFF_BUF1 - S::OFF_BUF0;
#define PVK_BUF(par) reinterpret_cast<float2 *>(smem + S::OFF_BUF0 + (int)(par) * BUF_STRIDE)
  float *famp = reinterpret_cast<float *>(smem + S::OFF_FAMP);
  // candidate list entry = bin | 0x8000 for a candidate that is not a local maximum (key 0); the
  // key is looked up in |fx|^2 through the bin
#define PVK_KEY(e) ((cbin[e] & 0x8000) ? 0u : __float_as_uint(famp[FA(cbin[e])]))
#define PVK_BIN(v) ((v) & 0x7fff)
  unsigned *hist = reinterpret_cast<unsigned *>(smem + S::OFF_HIST);   // 3 x 128 words (256 16-bit buckets each)
  double *redd = reinterpret_cast<double *>(smem + S::OFF_RED);
  float *redf = reinterpret_cast<float *>(smem + S::OFF_REDF);
  unsigned *redu = reinterpret_cast<unsigned *>(smem + S::OFF_REDU);
  int *wsA = reinterpret_cast<int *>(smem + S::OFF_WS);
  int *wsB = wsA + 32;
  unsigned short *cbin = reinterpret_cast<unsigned short *>(smem + S::OFF_CBIN);
  unsigned short *pk1 = reinterpret_cast<unsigned short *>(smem + S::OFF_PK);
  unsigned short *pk2 = pk1 + (prm.npks + 7) / 8 * 8;
  unsigned *selw = reinterpret_cast<unsigned *>(smem + S::OFF_SELW);   // selection / tie ballots, one word per 32 candidates
  unsigned *tiew = selw + M / 32;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t clip = blockIdx.x / prm.nruns;
  const int64_t run = blockIdx.x % prm.nruns;
  const int64_t r0 = run * prm.run;
  const int64_t r1 = (r0 + prm.run < prm.nframes) ? r0 + prm.run : prm.nframes;
  const float *xc = prm.x + clip * prm.clip_stride;
  const float2 *twp = prm.tables;
  const float2 *twr = prm.tables + P::TW_TOTAL;
  const int K = prm.npks;
  const double inv_2pidt = 1.0 / (prm.dt * 6.283185307179586), inv_dt = 1.0 / prm.dt;
  const double pi_fstep = 3.141592653589793 / prm.fstep;

  // ---- the run starts one row early: row r0 - 1 only leaves its spectrum behind (the "previous"
  //      spectrum of row r0) and emits nothing -- same code, one copy of the FFT in the instruction
  //      cache.  Global frame 0 has the all-zero previous spectrum instead (PVAnalysis.py:121).
  const bool zero_start = (r0 == 0 && prm.prev_zero);
  if (zero_start) {
    float2 *pb = PVK_BUF((r0 & 1) ^ 1);
    for (int i = tid; i < P::MP; i += T) pb[i] = make_float2(0.f, 0.f);
    __syncthreads();
  }
  for (int64_t r = zero_start ? r0 : r0 - 1; r < r1; ++r) {
    const bool emit = r >= r0;
    float2 *cur = PVK_BUF(r & 1);
    const float2 *prev = PVK_BUF((r & 1) ^ 1);
    const int64_t row = clip * prm.out_rows + r;
    {
      float2 ux[1 << P::lr(0)];
      frame_load<LOGM>(xc + (prm.frame0 + r) * (int64_t)prm.hop, ux);
      fft_frame_regs<LOGM>(ux, prm.win, twp, cur);
    }

    // ---- untangle -> fx[0..M), |fx|, min / max / sum of squares
    float lmin = 3.402823466e+38f, lmax = 0.f, lsum = 0.f;
    float2 *so = (prm.spec_out && emit) ? prm.spec_out + row * M : nullptr;
    constexpr int UI = (M / 2) / T;                            // pairs per thread (0: fewer pairs than threads)
#pragma unroll
    for (int it = 0; it < (UI > 0 ? UI : 1); ++it) {
      const int k = tid + it * T;
      if (UI == 0 && k >= M / 2) break;
      float2 xa, xb;
      if (it == 0 && k == 0) {
        const float2 z0 = cur[PADC(0)], zh = cur[PADC(M / 2)];
        xa = make_float2(z0.x + z0.y, 0.f);
        xb = make_float2(zh.x, -zh.y);
      } else {
        const float2 a = cur[PADC(k)], bq = cur[PADC(M - k)];
        const float2 e = make_float2(0.5f * (a.x + bq.x), 0.5f * (a.y - bq.y));
        const float2 o = make_float2(0.5f * (a.y + bq.y), -0.5f * (a.x - bq.x));
        const float2 wo = cmul(o, __ldg(twr + k));
        xa = make_float2(e.x + wo.x, e.y + wo.y);
        xb = make_float2(e.x - wo.x, -(e.y - wo.y));
      }
      const int kb = (k == 0) ? M / 2 : M - k;
      cur[PADC(k)] = xa;
      cur[PADC(kb)] = xb;
      // |fx|^2 in fp32 without FMA contraction (bit-identical to numpy float32 re*re + im*im).
      // Every comparison PeakFinder makes on |fx| is made on this power instead: fp64
      // sqrt is strictly increasing on distinct fp32 values, so the decisions are exactly
      // those on famp = sqrt(float64(power)) -- and no square root per bin is needed.
      const float pa = __fadd_rn(__fmul_rn(xa.x, xa.x), __fmul_rn(xa.y, xa.y));
      const float pb = __fadd_rn(__fmul_rn(xb.x, xb.x), __fmul_rn(xb.y, xb.y));
      famp[FA(k)] = pa;
      famp[FA(kb)] = pb;
      if (so) { so[k] = xa; so[kb] = xb; }
      lmin = fminf(lmin, fminf(pa, pb));
      lmax = fmaxf(lmax, fmaxf(pa, pb));
      lsum += pa + pb;
    }
    for (int w = tid; w < 3 * 128; w += T) hist[w] = 0u;        // the select's histograms (read after >= 2 barriers)
    {
      // powers are >= 0: their bit patterns order like the values, so one REDUX each
      const float wmin = __uint_as_float(warp_umin(__float_as_uint(lmin)));
      const float wmax = __uint_as_float(warp_umax(__float_as_uint(lmax)));
      const double wsum = warp_sum((double)lsum);
      if (lane == 0) { redf[warp] = wmin; redf[16 + warp] = wmax; redd[warp] = wsum; }
    }
    __syncthreads();
    if (!emit) continue;                                       // warm-up row: only its spectrum is needed
    float miny = redf[0], ymax = redf[16];
    double sumsq = redd[0];
#pragma unroll
    for (int w = 1; w < NW; ++w) {
      miny = fminf(miny, redf[w]);
      ymax = fmaxf(ymax, redf[16 + w]);
      sumsq += redd[w];
    }
    // PeakFinder.__init__ :57-70 and findpos :164,174 (miny / ymax are powers here)
    const double miny_d = sqrt((double)miny);
    double minamp = sqrt((double)ymax) * prm.pkthresh;
    if (minamp == 0.0) minamp = miny_d;
    const double th = minamp - miny_d;

    // ---- candidates: interior local maxima above threshold (or everything when th < 0),
    //      compacted in bin order into (cbin, ckey).  Thread t scans bins [t*CB, (t+1)*CB).
    //      The strict fp64 test (y - miny) > th is decided on the fp32 power outside a guard
    //      band of 2^-17 relative around minamp^2 (fp64 rounding moves either side by < 2^-50).
    int C = 0;
    unsigned lo = 0xffffffffu, hi = 0u;
    {
      const int kb0 = tid * CB;
      float y[CB + 2];
      if constexpr (CB % 4 == 0) {
#pragma unroll
        for (int j = 0; j < CB / 4; ++j) {
          const float4 v = *reinterpret_cast<const float4 *>(famp + FA(kb0 + 4 * j));
          y[4 * j + 1] = v.x; y[4 * j + 2] = v.y; y[4 * j + 3] = v.z; y[4 * j + 4] = v.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < CB; ++j) y[j + 1] = famp[FA(kb0 + j)];
      }
      y[0] = kb0 > 0 ? famp[FA(kb0 - 1)] : 0.f;
      y[CB + 1] = kb0 + CB < M ? famp[FA(kb0 + CB)] : 0.f;
      const bool allc = th < 0.0;
      float thr_hi = -1.f, thr_lo = -1.f;                      // th < 0: every local maximum passes
      if (!allc) {
        const float mf = (float)(minamp * minamp);
        thr_hi = mf * (1.f + 7.6293945e-6f); thr_lo = mf * (1.f - 7.6293945e-6f);
      }
      unsigned interior = (1u << CB) - 1u;                     // bins 1 .. M-2
      if (tid == 0) interior &= ~1u;
      if (tid == T - 1) interior &= ~(1u << (CB - 1));
      unsigned pbits = 0;                                      // local maxima not below the band
#pragma unroll
      for (int i = 0; i < CB; ++i) {
        const float yv = y[i + 1];
        if ((y[i] < yv) && (yv >= y[i + 2]) && !(yv < thr_lo)) pbits |= 1u << i;
      }
      pbits &= interior;
      unsigned kmin = 0xffffffffu, kmax = 0u;
      for (unsigned rem = pbits; rem;) {                       // few per thread: settle the band, key range
        const int i = __ffs((int)rem) - 1;
        rem &= rem - 1u;
        const float yv = famp[FA(kb0 + i)];
        bool c = yv > thr_hi;
        if (!c) c = (sqrt((double)yv) - miny_d) > th;
        if (c) {
          const unsigned key = __float_as_uint(yv);
          kmin = key < kmin ? key : kmin; kmax = key > kmax ? key : kmax;
        } else {
          pbits &= ~(1u << i);
        }
      }
      unsigned cbits = pbits;
      if (allc) {                                              // non-maxima are candidates too, key 0
        cbits = interior;
        if (interior & ~pbits) kmin = 0u;
      }
      const int cnt = __popc(cbits);
      const int incl = warp_scan_incl(cnt);
      kmin = warp_umin(kmin);
      kmax = warp_umax(kmax);
      if (lane == 31) redu[warp] = (unsigned)incl;
      if (lane == 0) { redu[16 + warp] = kmin; redu[32 + warp] = kmax; }
      __syncthreads();
      int pos = incl - cnt;
#pragma unroll
      for (int w = 0; w < NW; ++w) {
        const int cw = (int)redu[w];
        pos += (w < warp) ? cw : 0;
        C += cw;
        lo = redu[16 + w] < lo ? redu[16 + w] : lo;
        hi = redu[32 + w] > hi ? redu[32 + w] : hi;
      }
      for (unsigned rem = cbits; rem;) {
        const int i = __ffs((int)rem) - 1;
        rem &= rem - 1u;
        cbin[pos] = (unsigned short)((kb0 + i) | (((pbits >> i) & 1u) ? 0 : 0x8000));
        ++pos;
      }
    }
    __syncthreads();

    // ---- top-K by (key desc, bin asc): exact radix select of the K-th largest key, 8 bits per
    //      level.  One barrier per level: all threads fill a 256-bucket histogram (16-bit counters,
    //      two per word), then EVERY warp scans it (same result in each, no broadcast through shared
    //      memory).  Three histograms rotate; all are zero at this point (cleared during the
    //      untangle) and level L >= 2 clears the one level L + 1 will use, whose last readers (the
    //      scans of level L - 2) finished before the barrier of level L - 1.
    int rr = K;
    bool exact_ties = false;
    const bool need_sel = C > K;
    if (need_sel) {
      for (int level = 0; level < 4; ++level) {
        unsigned *h = hist + (level % 3) * 128;
        const unsigned range = hi - lo;
        const int bl = 32 - __clz((int)range);
        const int sh = bl > 8 ? bl - 8 : 0;
        for (int e = tid; e < C; e += T) {
          const unsigned key = PVK_KEY(e);
          if (key >= lo && key <= hi) {
            const unsigned b = (key - lo) >> sh;
            atomicAdd(&h[b >> 1], 1u << ((b & 1u) * 16u));
          }
        }
        if (level >= 2) {
          unsigned *hn = hist + ((level + 1) % 3) * 128;
          for (int w = tid; w < 128; w += T) hn[w] = 0u;
        }
        __syncthreads();
        // lane l owns buckets 255 - 8 l - q, q = 0 .. 7 (descending keys) = words 127 - 4 l - j, high half first
        int c[8], sum = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const unsigned w = h[127 - 4 * lane - j];
          c[2 * j] = (int)(w >> 16); c[2 * j + 1] = (int)(w & 0xffffu);
          sum += c[2 * j] + c[2 * j + 1];
        }
        const int incl = warp_scan_incl(sum);
        int above = incl - sum;
        const bool mine = above < rr && rr <= incl;               // exactly one lane
        int bq = 0, ab = 0, cq = 0;
        if (mine) {
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            if (above < rr && rr <= above + c[q]) { bq = 255 - 8 * lane - q; ab = above; cq = c[q]; }
            above += c[q];
          }
        }
        const int src = __ffs((int)__ballot_sync(FULL, mine)) - 1;
        const int b = __shfl_sync(FULL, bq, src), nabove = __shfl_sync(FULL, ab, src), cb = __shfl_sync(FULL, cq, src);
        lo = lo + ((unsigned)b << sh);
        const unsigned hi2 = lo + ((1u << sh) - 1u);
        hi = hi2 < hi ? hi2 : hi;
        rr -= nabove;
        if (cb == rr) break;
        if (sh == 0) { exact_ties = true; break; }
      }
    }

    // ---- selected entries, compacted in bin order into pk1.  Selected = key above the boundary
    //      bucket, or inside it (only its first rr entries in bin order when the bucket is a run of
    //      exactly equal keys).  Entry e = round * T + tid; the warps' ballots go to shared memory
    //      (word q = e / 32), ONE barrier, then the position of an entry is the number of set bits
    //      before it (a warp scan over the words).
    const unsigned short *sel = cbin;
    int ns = C;
    if (need_sel) {
      constexpr int NCH = (M + 1023) / 1024;                       // chunks of 32 mask words
      const int nwords = (C + 31) >> 5;
      // exclusive prefix of the set bits of words[0 .. nwords): value for word q in lane q % 32 of chunk q / 32
      auto word_prefix = [&](const unsigned *words, int (&excl)[NCH]) -> int {
        int total = 0;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          const int q = c * 32 + lane;
          const int v = q < nwords ? __popc(words[q]) : 0;
          const int incl = warp_scan_incl(v);
          excl[c] = total + incl - v;
          total += __shfl_sync(FULL, incl, 31);
        }
        return total;
      };
      auto prefix_of = [&](const int (&excl)[NCH], int q) -> int {
        int val = 0;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          const int t = __shfl_sync(FULL, excl[c], q & 31);
          if ((q >> 5) == c) val = t;
        }
        return val;
      };
      unsigned flags = 0, ties = 0;                                // bit j: my entry of round j is selected / a tie
      for (int e0 = 0, j = 0; e0 < C; e0 += T, ++j) {
        const int e = e0 + tid;
        const unsigned key = e < C ? PVK_KEY(e) : 0u;
        const bool inA = e < C && key > hi;
        const bool inB = e < C && key >= lo && key <= hi;
        const bool s = inA || (inB && !exact_ties);
        const unsigned ms = __ballot_sync(FULL, s), mt = __ballot_sync(FULL, inB);
        if (lane == 0) { selw[(e0 >> 5) + warp] = ms; tiew[(e0 >> 5) + warp] = mt; }
        if (s) flags |= 1u << j;
        if (inB) ties |= 1u << j;
      }
      __syncthreads();
      if (exact_ties) {                                            // rare: the first rr ties in bin order join
        int excl[NCH];
        word_prefix(tiew, excl);
        for (int e0 = 0, j = 0; e0 < C; e0 += T, ++j) {
          const int q = (e0 >> 5) + warp;
          const int tpos = prefix_of(excl, q) + __popc(tiew[q < nwords ? q : 0] & lanemask_lt());
          const bool s = ((ties >> j) & 1u) && tpos < rr;
          const unsigned ms = __ballot_sync(FULL, s);
          if (lane == 0 && q < nwords) atomicOr(&selw[q], ms);
          if (s) flags |= 1u << j;
        }
        __syncthreads();
      }
      {
        int excl[NCH];
        word_prefix(selw, excl);
        for (int e0 = 0, j = 0; e0 < C; e0 += T, ++j) {
          const int q = (e0 >> 5) + warp;
          const int pos = prefix_of(excl, q) + __popc(selw[q < nwords ? q : 0] & lanemask_lt());
          if ((flags >> j) & 1u) pk1[pos] = PVK_BIN(cbin[e0 + tid]);
        }
      }
      sel = pk1;
      ns = K;
      __syncthreads();
    }

    // ---- salience filter, rad = 5 (PeakFinder.py:113-134 as called at PVAnalysis.py:177), one
    //      thread per selected peak; survivors compacted in bin order into pk2
    int nk = 0;
    for (int e0 = 0, round = 0; e0 < ns; e0 += T, ++round) {
      const int e = e0 + tid;
      bool keep = false;
      int k = 0;
      if (e < ns) {
        k = PVK_BIN(sel[e]);
        const float y = famp[FA(k)];
        const int a = k - 5 > 1 ? k - 5 : 1, b = k + 5 < M - 1 ? k + 5 : M - 1;
        keep = true;
        for (int m = a; m <= b; ++m) keep = keep && !(famp[FA(m)] > y);
      }
      const int pos = round_pos<NW>(keep, wsA, round, nk);
      if (keep) pk2[pos] = (unsigned short)k;
    }
    __syncthreads();
    const unsigned short *pk = pk2;

    // ---- per-peak epilogue, freq > 0 filter, ordered write of the zero padded row
    const int64_t ob = row * K;
    int outbase = 0;
    for (int p0 = 0, round = 0; p0 < nk; p0 += T, ++round) {
      const int p = p0 + tid;
      PeakVals v;
      bool valid = false;
      int k = 0;
      if (p < nk) {
        k = pk[p];
        valid = peak_epilogue(k, M, cur, prev, FampPow{famp}, prm.fbin, prm.wfbin, prm.dt, inv_2pidt, inv_dt, pi_fstep, v);
      }
      const int64_t pos = ob + round_pos<NW>(valid, wsB, round, outbase);
      if (valid) {
        prm.f[pos] = v.f; prm.mag[pos] = v.mag; prm.ph[pos] = v.ph;
        prm.realph[pos] = v.realph; prm.binno[pos] = (double)k;
        if (prm.fine_pos) {
          double fp, fv;
          refine_peak(k, FampPow{famp}, fp, fv);
          prm.fine_pos[pos] = fp; prm.fine_val[pos] = fv;
        }
      }
    }
    for (int p = outbase + tid; p < K; p += T) {
      prm.f[ob + p] = 0.0; prm.mag[ob + p] = 0.0; prm.ph[ob + p] = 0.0;
      prm.realph[ob + p] = 0.0; prm.binno[ob + p] = 0.0;
      if (prm.fine_pos) { prm.fine_pos[ob + p] = 0.0; prm.fine_val[ob + p] = 0.0; }
    }
    if (tid == 0) {
      prm.npk[row] = outbase;
      prm.totalmag[row] = sqrt(sumsq);                       // PVAnalysis.py:210
    }
    __syncthreads();   // prev buffer is overwritten by the next frame's FFT
  }
  (void)N;
}

// ------------------------------------------------------------------ one warp per frame (LOGM 9, 10)
// analyze_warp_kernel: a CTA of W warps walks a run of frames W at a time, warp w taking local frame
// t = g W + w of group g (t = 0 is the warm-up row r0 - 1).  A frame never leaves its warp: the FFT
// exchanges, the reductions, the select and the compactions use __syncwarp, shuffles and ballots.
// The spectra live in a ring of W + 1 slots, frame t in slot t mod (W + 1); the only data shared
// between warps is the previous frame's untangled spectrum that a frame's epilogue reads.  Two
// block barriers per group: A, after the group's untangles and selects (frame t's epilogue reads
// slot t - 1, which warp w - 1 wrote), and B, after the group's epilogues (each of them reads its
// own slot and the one before, and the next group overwrites every slot but the last one written).
// Every value is computed as analyze_kernel<LOGM> computes it, so the outputs are bit-identical:
//   - the FFT runs Plan<LOGM>'s passes, twiddles and butterflies; lane l takes the butterflies
//     i = l, l + 32, ... of each pass (two of the 64-thread plan's threads per lane);
//   - the untangle keeps the 64-thread partition of the bins (virtual thread v = l + 32 h, h = 0, 1)
//     because totalmag sums the fp32 partial sums of those threads per warp in fp64, then adds the
//     two warp sums;
//   - the powers are not stored: every reader recomputes them from the spectrum (bin_power);
//   - candidates, radix select, tie rule, salience and epilogue decide exactly as there.
// analyze_kernel's FFT and untangle are written with plain fp32 products and sums, and the compiler
// fuses products into FFMA at its own discretion, site by site and depending on the kernel around
// them.  The warp kernel spells out the roundings analyze_kernel<9/10> was compiled to (read off its
// SASS), so that its spectrum has the same bits:
//   - twiddle products of the exchange passes: re = a.x w.x (exact) - rn(a.y w.y), im = a.y w.x
//     (exact) + rn(a.x w.y); of the untangle: re = o.x w.x - rn(o.y w.y), im = o.x w.y + rn(o.y w.x);
//   - mul_w16 cases 1, 3, 5, 7: the first product exact, the second rounded; case 6 rounded; the
//     case-2 products (d.x + d.y) C8 and (d.y - d.x) C8 stay exact into both sums of the next stage;
//   - first pass: the windowed upper half of each first-stage butterfly is rounded, the lower half exact.
// The fused multiply-add of those roundings.  The emulator build (g++ -ffp-contract=off) fuses no
// product anywhere, so there it is unfused too: the emulator's analysis spectra then stay those of
// its analyze_kernel, bank_kernel and harmonic_kernel builds.
__device__ __forceinline__ float wfma(float a, float b, float c) {
#ifdef PVK_EMU
  return __fadd_rn(__fmul_rn(a, b), c);
#else
  return fmaf(a, b, c);
#endif
}
__device__ __forceinline__ float2 wcmul_pass(float2 a, float2 w) {
  return make_float2(wfma(a.x, w.x, -__fmul_rn(a.y, w.y)), wfma(a.y, w.x, __fmul_rn(a.x, w.y)));
}
__device__ __forceinline__ float2 wcmul_untangle(float2 o, float2 w) {
  return make_float2(wfma(o.x, w.x, -__fmul_rn(o.y, w.y)), wfma(o.x, w.y, __fmul_rn(o.y, w.x)));
}
__device__ __forceinline__ float wsub(float a, float b) { return __fadd_rn(a, -b); }

// dft_dif<LR> with those roundings.  WIN: u holds raw samples, w the window (first pass).
template <int LR, bool WIN> __device__ __forceinline__ void wdft_dif(float2 *u, const float2 *w) {
  constexpr int R = 1 << LR;
  const float C8 = 0.70710678118654752440f, C1 = 0.92387953251128675613f, S1 = 0.38268343236508977173f;
  unsigned pend = 0;                                         // u[i] holds s with value s * C8, unrounded
#pragma unroll
  for (int h = R / 2; h >= 1; h >>= 1) {
    unsigned npend = 0;
#pragma unroll
    for (int g = 0; g < R; g += 2 * h) {
#pragma unroll
      for (int j = 0; j < h; ++j) {
        const int ia = g + j, ib = g + j + h;
        const float2 a = u[ia], b = u[ib];
        float2 sm, d;
        if (WIN && h == R / 2) {
          const float2 pb = make_float2(__fmul_rn(b.x, w[ib].x), __fmul_rn(b.y, w[ib].y));
          sm = make_float2(wfma(a.x, w[ia].x, pb.x), wfma(a.y, w[ia].y, pb.y));
          d = make_float2(wfma(a.x, w[ia].x, -pb.x), wfma(a.y, w[ia].y, -pb.y));
        } else if ((pend >> ia) & 1u) {
          sm = make_float2(wfma(a.x, C8, b.x), wfma(a.y, C8, b.y));
          d = make_float2(wfma(a.x, C8, -b.x), wfma(a.y, C8, -b.y));
        } else if ((pend >> ib) & 1u) {
          sm = make_float2(wfma(b.x, C8, a.x), wfma(b.y, C8, a.y));
          d = make_float2(wfma(-b.x, C8, a.x), wfma(-b.y, C8, a.y));
        } else {
          sm = make_float2(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y));
          d = make_float2(wsub(a.x, b.x), wsub(a.y, b.y));
        }
        u[ia] = sm;
        switch (j * (8 / h)) {
          case 0: u[ib] = d; break;
          case 4: u[ib] = make_float2(d.y, -d.x); break;
          case 2: u[ib] = make_float2(__fadd_rn(d.x, d.y), wsub(d.y, d.x)); npend |= 1u << ib; break;
          case 6: u[ib] = make_float2(__fmul_rn(wsub(d.y, d.x), C8), -__fmul_rn(__fadd_rn(d.x, d.y), C8)); break;
          case 1: u[ib] = make_float2(wfma(d.x, C1, __fmul_rn(d.y, S1)), wfma(d.y, C1, -__fmul_rn(d.x, S1))); break;
          case 3: u[ib] = make_float2(wfma(d.x, S1, __fmul_rn(d.y, C1)), wfma(d.y, S1, -__fmul_rn(d.x, C1))); break;
          case 5: u[ib] = make_float2(wfma(d.y, C1, -__fmul_rn(d.x, S1)), wfma(-d.y, S1, -__fmul_rn(d.x, C1))); break;
          default: u[ib] = make_float2(wfma(d.y, S1, -__fmul_rn(d.x, C1)), wfma(-d.y, C1, -__fmul_rn(d.x, S1))); break;
        }
      }
    }
    pend = npend;
  }
}

template <int LOGM, int Q> struct WPass {
  using P = Plan<LOGM>;
  static constexpr int M = P::M;
  static constexpr int LR = P::lr(Q), R = 1 << LR, PP = 1 << P::lp(Q);
  static constexpr int NBF = M >> LR, NBL = NBF / 32;        // butterflies per lane
  static constexpr int OFF = P::tw_off(Q);
  static_assert(NBF % 32 == 0, "whole butterflies per lane");

  static __device__ __forceinline__ void run(const float2 *__restrict__ twp, float2 *buf) {
    const int lane = lane_id();
    // in place: every input of the lane's butterflies is read before any output lands.  Each
    // butterfly is twiddled and transformed as soon as it is read, so that no twiddle stays live
    // beside the 2 x 16 points of a radix-16 pass.
    float2 u[NBL][R];
#pragma unroll
    for (int b = 0; b < NBL; ++b) {
      const int i = lane + 32 * b;
      const int k = i & (PP - 1);
      u[b][0] = buf[PADC(i)];
#pragma unroll
      for (int r = 1; r < R; ++r) u[b][r] = wcmul_pass(buf[PADC(i + r * NBF)], __ldg(twp + OFF + (r - 1) * PP + k));
      wdft_dif<LR, false>(u[b], nullptr);
    }
    __syncwarp();
#pragma unroll
    for (int b = 0; b < NBL; ++b) {
      const int i = lane + 32 * b;
      const int k = i & (PP - 1);
      const int j = ((i - k) << LR) + k;
#pragma unroll
      for (int s = 0; s < R; ++s) buf[PADC(j + s * PP)] = u[b][brev<LR>(s)];
    }
    __syncwarp();
    if constexpr (Q + 1 < P::NPASS) WPass<LOGM, Q + 1>::run(twp, buf);
  }
};

// framing + window + first pass straight from the signal, then the exchange passes; natural order in buf
template <int LOGM>
__device__ __forceinline__ void wfft_frame(const float *__restrict__ xf, const float *__restrict__ win,
                                           const float2 *__restrict__ twp, float2 *buf) {
  using P = Plan<LOGM>;
  constexpr int M = P::M, LR = P::lr(0), R = 1 << LR, NBF = M >> LR;
  static_assert(NBF % 32 == 0, "whole butterflies per lane");
  const int lane = lane_id();
  const bool al8 = ((reinterpret_cast<uintptr_t>(xf) & 7) == 0);
#pragma unroll
  for (int b = 0; b < NBF / 32; ++b) {
    const int i = lane + 32 * b;
    float2 u[R], wv[R];
#pragma unroll
    for (int r = 0; r < R; ++r) u[r] = ldg_stream2(xf + 2 * (i + r * NBF), al8);
#pragma unroll
    for (int r = 0; r < R; ++r) wv[r] = __ldg(reinterpret_cast<const float2 *>(win) + i + r * NBF);
    wdft_dif<LR, true>(u, wv);
#pragma unroll
    for (int s = 0; s < R; ++s) buf[PADC(i * R + s)] = u[brev<LR>(s)];
  }
  __syncwarp();
  if constexpr (P::NPASS > 1) WPass<LOGM, 1>::run(twp, buf);
}

// Warps per CTA.  W + 1 spectrum slots plus W scratch areas: 98.9 KB at LOGM 10 (two CTAs = 16
// warps per SM, as many as 128 registers per thread allow), 51.5 KB at LOGM 9.
constexpr int AW = 8;

template <int LOGM> struct WSmem {
  using P = Plan<LOGM>;
  static constexpr int SLOT = P::MP * 8;                     // one padded spectrum
  static constexpr int OFF_SCR = (AW + 1) * SLOT;
  // per warp: the candidate list (uint16), compacted in place into the selection and then into the
  // salience survivors (a compaction never moves an entry up), and one 256-bucket histogram
  static constexpr int SCR = P::M * 2 + 128 * 4;
  static constexpr int BYTES = OFF_SCR + AW * SCR;
};

// Peak picking of one frame by one warp on its untangled spectrum `cur` (PeakFinder.__init__
// :57-70, findpos, salience :113-134): the same decisions as analyze_kernel, with warp scans and
// ballots instead of block barriers.  Leaves the surviving bins, ascending, in pk[0, return value).
template <int LOGM>
__device__ __forceinline__ int warp_peaks(const float2 *cur, float miny, float ymax, double pkthresh, int K,
                                          unsigned short *pk, unsigned *hist) {
  constexpr int M = Plan<LOGM>::M;
  constexpr int CB = M / 32;                                 // contiguous bins per lane in the candidate scan
  constexpr unsigned CB_MASK = CB == 32 ? 0xffffffffu : (1u << CB) - 1u;
  const SpecPow pw{cur};
  const int lane = lane_id();
  unsigned short *cbin = pk;
  // candidate list entry = bin | 0x8000 for a candidate that is not a local maximum (key 0)
#define PVK_WKEY(v) (((v) & 0x8000) ? 0u : __float_as_uint(pw(v)))
  const double miny_d = sqrt((double)miny);
  double minamp = sqrt((double)ymax) * pkthresh;
  if (minamp == 0.0) minamp = miny_d;
  const double th = minamp - miny_d;

  // ---- candidates: interior local maxima above threshold (or everything when th < 0), compacted in
  //      bin order.  Lane l scans bins [l CB, (l + 1) CB); the guard band as in analyze_kernel.
  int C;
  unsigned lo, hi;
  {
    const int kb0 = lane * CB;
    const bool allc = th < 0.0;
    float thr_hi = -1.f, thr_lo = -1.f;                      // th < 0: every local maximum passes
    if (!allc) {
      const float mf = (float)(minamp * minamp);
      thr_hi = mf * (1.f + 7.6293945e-6f); thr_lo = mf * (1.f - 7.6293945e-6f);
    }
    unsigned interior = CB_MASK;                             // bins 1 .. M-2
    if (lane == 0) interior &= ~1u;
    if (lane == 31) interior &= ~(1u << (CB - 1));
    unsigned pbits = 0;                                      // local maxima not below the band
    float yl = kb0 > 0 ? pw(kb0 - 1) : 0.f, yv = pw(kb0);
#pragma unroll
    for (int i = 0; i < CB; ++i) {
      const float yr = (i + 1 < CB || kb0 + CB < M) ? pw(kb0 + i + 1) : 0.f;
      if ((yl < yv) && (yv >= yr) && !(yv < thr_lo)) pbits |= 1u << i;
      yl = yv; yv = yr;
    }
    pbits &= interior;
    unsigned kmin = 0xffffffffu, kmax = 0u;
    for (unsigned rem = pbits; rem;) {                       // few per lane: settle the band, key range
      const int i = __ffs((int)rem) - 1;
      rem &= rem - 1u;
      const float y = pw(kb0 + i);
      bool c = y > thr_hi;
      if (!c) c = (sqrt((double)y) - miny_d) > th;
      if (c) {
        const unsigned key = __float_as_uint(y);
        kmin = key < kmin ? key : kmin; kmax = key > kmax ? key : kmax;
      } else {
        pbits &= ~(1u << i);
      }
    }
    unsigned cbits = pbits;
    if (allc) {                                              // non-maxima are candidates too, key 0
      cbits = interior;
      if (interior & ~pbits) kmin = 0u;
    }
    const int cnt = __popc(cbits);
    const int incl = warp_scan_incl(cnt);
    C = __shfl_sync(FULL, incl, 31);
    lo = warp_umin(kmin);
    hi = warp_umax(kmax);
    int pos = incl - cnt;
    for (unsigned rem = cbits; rem;) {
      const int i = __ffs((int)rem) - 1;
      rem &= rem - 1u;
      cbin[pos++] = (unsigned short)((kb0 + i) | (((pbits >> i) & 1u) ? 0 : 0x8000));
    }
    __syncwarp();
  }

  // ---- top-K by (key desc, bin asc): exact radix select of the K-th largest key, 8 bits per level,
  //      as in analyze_kernel; every lane clears the histogram words it reads
  int rr = K;
  bool exact_ties = false;
  const bool need_sel = C > K;
  if (need_sel) {
    for (int level = 0; level < 4; ++level) {
      const unsigned range = hi - lo;
      const int bl = 32 - __clz((int)range);
      const int sh = bl > 8 ? bl - 8 : 0;
      for (int e = lane; e < C; e += 32) {
        const unsigned key = PVK_WKEY(cbin[e]);
        if (key >= lo && key <= hi) {
          const unsigned b = (key - lo) >> sh;
          atomicAdd(&hist[b >> 1], 1u << ((b & 1u) * 16u));
        }
      }
      __syncwarp();
      // lane l owns buckets 255 - 8 l - q, q = 0 .. 7 (descending keys) = words 127 - 4 l - j, high half first
      int c[8], sum = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const unsigned w = hist[127 - 4 * lane - j];
        hist[127 - 4 * lane - j] = 0u;
        c[2 * j] = (int)(w >> 16); c[2 * j + 1] = (int)(w & 0xffffu);
        sum += c[2 * j] + c[2 * j + 1];
      }
      __syncwarp();
      const int incl = warp_scan_incl(sum);
      int above = incl - sum;
      const bool mine = above < rr && rr <= incl;               // exactly one lane
      int bq = 0, ab = 0, cq = 0;
      if (mine) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          if (above < rr && rr <= above + c[q]) { bq = 255 - 8 * lane - q; ab = above; cq = c[q]; }
          above += c[q];
        }
      }
      const int src = __ffs((int)__ballot_sync(FULL, mine)) - 1;
      const int b = __shfl_sync(FULL, bq, src), nabove = __shfl_sync(FULL, ab, src), cb = __shfl_sync(FULL, cq, src);
      lo = lo + ((unsigned)b << sh);
      const unsigned hi2 = lo + ((1u << sh) - 1u);
      hi = hi2 < hi ? hi2 : hi;
      rr -= nabove;
      if (cb == rr) break;
      if (sh == 0) { exact_ties = true; break; }
    }

    // ---- selected entries, compacted in place in bin order.  Selected = key above the boundary
    //      bucket, or inside it (only its first rr entries in bin order when the bucket is a run of
    //      exactly equal keys).  An entry's position is at most its index, and the entries of a
    //      round are read before its ballot, so no entry is overwritten before it is read.
    int sbase = 0, tbase = 0;
    for (int e0 = 0; e0 < C; e0 += 32) {
      const int e = e0 + lane;
      const unsigned v = e < C ? cbin[e] : 0u;
      const unsigned key = e < C ? PVK_WKEY(v) : 0u;
      const bool inA = e < C && key > hi;
      const bool inB = e < C && key >= lo && key <= hi;
      bool s = inA || inB;
      if (exact_ties) {                                          // rare: the first rr ties in bin order join
        const unsigned mt = __ballot_sync(FULL, inB);
        s = inA || (inB && tbase + __popc(mt & lanemask_lt()) < rr);
        tbase += __popc(mt);
      }
      const unsigned ms = __ballot_sync(FULL, s);
      if (s) cbin[sbase + __popc(ms & lanemask_lt())] = (unsigned short)(v & 0x7fff);
      sbase += __popc(ms);
    }
    __syncwarp();
  }
  const int ns = need_sel ? K : C;

  // ---- salience filter, rad = 5 (PeakFinder.py:113-134 as called at PVAnalysis.py:177), one lane
  //      per selected peak; survivors compacted in place in bin order
  int nk = 0;
  for (int e0 = 0; e0 < ns; e0 += 32) {
    const int e = e0 + lane;
    bool keep = false;
    int k = 0;
    if (e < ns) {
      k = cbin[e] & 0x7fff;
      const float y = pw(k);
      const int a = k - 5 > 1 ? k - 5 : 1, b = k + 5 < M - 1 ? k + 5 : M - 1;
      keep = true;
      for (int m = a; m <= b; ++m) keep = keep && !(pw(m) > y);
    }
    const unsigned mk = __ballot_sync(FULL, keep);
    if (keep) cbin[nk + __popc(mk & lanemask_lt())] = (unsigned short)k;
    nk += __popc(mk);
  }
  __syncwarp();
#undef PVK_WKEY
  return nk;
}

template <int LOGM>
__global__ void __launch_bounds__(AW * 32, 16 / AW) analyze_warp_kernel(AParams prm) {
  using P = Plan<LOGM>;
  using S = WSmem<LOGM>;
  constexpr int M = P::M, VT = P::T, W = AW;
  static_assert(VT == 64, "totalmag follows the 64-thread partition of analyze_kernel<LOGM>");
  PVK_SMEM(smem);
#define PVK_SLOT(s) reinterpret_cast<float2 *>(smem + (int)(s) * S::SLOT)
  const int lane = lane_id(), warp = warp_id();
  unsigned short *cbin = reinterpret_cast<unsigned short *>(smem + S::OFF_SCR + warp * S::SCR);
  unsigned *hist = reinterpret_cast<unsigned *>(cbin + M);  // 128 words (256 16-bit buckets)

  const int64_t clip = blockIdx.x / prm.nruns;
  const int64_t run = blockIdx.x % prm.nruns;
  const int64_t r0 = run * prm.run;
  const int64_t r1 = (r0 + prm.run < prm.nframes) ? r0 + prm.run : prm.nframes;
  const int K = prm.npks;
  const bool zero_start = (r0 == 0 && prm.prev_zero);
  // local frame t = r - (r0 - 1): t = 0 only leaves its spectrum behind (the warm-up row, or the
  // all-zero previous spectrum of global frame 0, PVAnalysis.py:121)
  const float *x0 = prm.x + clip * prm.clip_stride + (prm.frame0 + r0 - 1) * (int64_t)prm.hop;   // frame t = 0
  const int64_t row0 = clip * prm.out_rows + r0 - 1;
  const int nloc = (int)(r1 - r0) + 1;

  // every level of the select reads its histogram and clears it: zero once, zero after every frame
#pragma unroll
  for (int j = 0; j < 4; ++j) hist[lane + 32 * j] = 0u;
  __syncwarp();

  int slot = warp;                                           // t mod (W + 1)
  for (int g0 = 0; g0 < nloc; g0 += W, slot = slot == 0 ? W : slot - 1) {
    const int t = g0 + warp;
    const bool act = t < nloc, emit = act && t > 0;
    const int64_t row = row0 + t;
    float2 *cur = PVK_SLOT(slot);
    const float2 *prev = PVK_SLOT(slot == 0 ? W : slot - 1);
    double sumsq = 0.0;
    int nk = 0;
    if (act && t == 0 && zero_start) {
      for (int i = lane; i < P::MP; i += 32) cur[i] = make_float2(0.f, 0.f);
    } else if (act) {
      wfft_frame<LOGM>(x0 + t * (int64_t)prm.hop, prm.win, prm.tables, cur);

      // ---- untangle -> fx[0..M), min / max / sum of the powers (bins of virtual thread v = lane + 32 h)
      float lmin = 3.402823466e+38f, lmax = 0.f, lsum[2] = {0.f, 0.f};
      float2 *so = (prm.spec_out && emit) ? prm.spec_out + row * M : nullptr;
      constexpr int UI = (M / 2) / VT;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
#pragma unroll
        for (int it = 0; it < UI; ++it) {
          const int k = lane + 32 * h + it * VT;
          float2 xa, xb;
          if (h == 0 && it == 0 && k == 0) {
            const float2 z0 = cur[PADC(0)], zh = cur[PADC(M / 2)];
            xa = make_float2(z0.x + z0.y, 0.f);
            xb = make_float2(zh.x, -zh.y);
          } else {
            const float2 a = cur[PADC(k)], bq = cur[PADC(M - k)];
            // (the products by 0.5 are exact: fused or not, the same bits)
            const float2 e = make_float2(__fmul_rn(0.5f, __fadd_rn(a.x, bq.x)), __fmul_rn(0.5f, wsub(a.y, bq.y)));
            const float2 o = make_float2(__fmul_rn(0.5f, __fadd_rn(a.y, bq.y)), __fmul_rn(-0.5f, wsub(a.x, bq.x)));
            const float2 wo = wcmul_untangle(o, __ldg(prm.tables + P::TW_TOTAL + k));
            xa = make_float2(__fadd_rn(e.x, wo.x), __fadd_rn(e.y, wo.y));
            xb = make_float2(wsub(e.x, wo.x), -wsub(e.y, wo.y));
          }
          const int kb = (k == 0) ? M / 2 : M - k;
          cur[PADC(k)] = xa;
          cur[PADC(kb)] = xb;
          const float pa = bin_power(xa), pb = bin_power(xb);
          if (so) { so[k] = xa; so[kb] = xb; }
          lmin = fminf(lmin, fminf(pa, pb));
          lmax = fmaxf(lmax, fmaxf(pa, pb));
          lsum[h] += pa + pb;
        }
      }
      // powers are >= 0: their bit patterns order like the values, so one REDUX each
      const float miny = __uint_as_float(warp_umin(__float_as_uint(lmin)));
      const float ymax = __uint_as_float(warp_umax(__float_as_uint(lmax)));
      sumsq = warp_sum((double)lsum[0]);
      sumsq += warp_sum((double)lsum[1]);
      __syncwarp();                                          // the untangled spectrum, for every lane
      if (emit) nk = warp_peaks<LOGM>(cur, miny, ymax, prm.pkthresh, K, cbin, hist);
    }
    __syncthreads();                                         // A: slot t - 1 holds frame t - 1's spectrum

    // ---- per-peak epilogue, freq > 0 filter, ordered write of the zero padded row
    if (emit) {
      const SpecPow pw{cur};
      const double inv_2pidt = 1.0 / (prm.dt * 6.283185307179586), inv_dt = 1.0 / prm.dt;
      const double pi_fstep = 3.141592653589793 / prm.fstep;
      const int64_t ob = row * K;
      int outbase = 0;
      for (int p0 = 0; p0 < nk; p0 += 32) {
        const int p = p0 + lane;
        PeakVals v;
        bool valid = false;
        int k = 0;
        if (p < nk) {
          k = cbin[p];
          valid = peak_epilogue(k, M, cur, prev, pw, prm.fbin, prm.wfbin, prm.dt, inv_2pidt, inv_dt, pi_fstep, v);
        }
        const unsigned m = __ballot_sync(FULL, valid);
        const int64_t pos = ob + outbase + __popc(m & lanemask_lt());
        outbase += __popc(m);
        if (valid) {
          prm.f[pos] = v.f; prm.mag[pos] = v.mag; prm.ph[pos] = v.ph;
          prm.realph[pos] = v.realph; prm.binno[pos] = (double)k;
          if (prm.fine_pos) {
            double fp, fv;
            refine_peak(k, pw, fp, fv);
            prm.fine_pos[pos] = fp; prm.fine_val[pos] = fv;
          }
        }
      }
      for (int p = outbase + lane; p < K; p += 32) {
        prm.f[ob + p] = 0.0; prm.mag[ob + p] = 0.0; prm.ph[ob + p] = 0.0;
        prm.realph[ob + p] = 0.0; prm.binno[ob + p] = 0.0;
        if (prm.fine_pos) { prm.fine_pos[ob + p] = 0.0; prm.fine_val[ob + p] = 0.0; }
      }
      if (lane == 0) {
        prm.npk[row] = outbase;
        prm.totalmag[row] = sqrt(sumsq);                     // PVAnalysis.py:210
      }
    }
    __syncthreads();                                         // B: the next group overwrites this group's slots
  }
#undef PVK_SLOT
}

// ------------------------------------------------------------------ f0-guided analysis
// PVHarmonic.run_pv / calc_pv_frame (PVAnalysis.py:419-538): same framing / FFT / phase
// difference as analyze_kernel, but the bins are read at multiples of a given f0 instead of
// being peak-picked.  One CTA walks a run of frames; the "previous spectrum" is that of the
// last PROCESSED frame (f0 > 0 and not NaN, :509), as the reference only replaces oldfft there
// (:491) -- a run starts by searching backwards for it.
struct HParams {
  const float *x;
  const float *win;
  const float2 *tables;
  const double *fbin;
  const double *wfbin;
  const double *f0;
  int hop, npks;
  double dt, sr, fmin;
  int64_t nframes;
  int run;
  double *f, *mag, *ph, *residual;
  int32_t *nharm;
};

__device__ __forceinline__ bool f0_valid(double v) { return v > 0.0; }   // false for NaN too (:509)

template <int LOGM>
__device__ __forceinline__ void untangle_power(float2 *cur, float *famp, const float2 *__restrict__ twr, bool power,
                                               double &lsum) {
  using P = Plan<LOGM>;
  constexpr int M = P::M, T = P::T;
  const int tid = threadIdx.x;
  for (int k = tid; k < M / 2; k += T) {
    float2 xa, xb;
    if (k == 0) {
      const float2 z0 = cur[PADC(0)], zh = cur[PADC(M / 2)];
      xa = make_float2(z0.x + z0.y, 0.f);
      xb = make_float2(zh.x, -zh.y);
    } else {
      const float2 a = cur[PADC(k)], bq = cur[PADC(M - k)];
      const float2 e = make_float2(0.5f * (a.x + bq.x), 0.5f * (a.y - bq.y));
      const float2 o = make_float2(0.5f * (a.y + bq.y), -0.5f * (a.x - bq.x));
      const float2 wo = cmul(o, __ldg(twr + k));
      xa = make_float2(e.x + wo.x, e.y + wo.y);
      xb = make_float2(e.x - wo.x, -(e.y - wo.y));
    }
    const int kb = (k == 0) ? M / 2 : M - k;
    cur[PADC(k)] = xa;
    cur[PADC(kb)] = xb;
    if (power) {
      const float pa = __fadd_rn(__fmul_rn(xa.x, xa.x), __fmul_rn(xa.y, xa.y));
      const float pb = __fadd_rn(__fmul_rn(xb.x, xb.x), __fmul_rn(xb.y, xb.y));
      famp[FA(k)] = pa;
      famp[FA(kb)] = pb;
      lsum += (double)pa + (double)pb;
    }
  }
}

// bin of harmonic i (0-based): np.round(np.arange(f0bin, M-1, f0bin))[i] = rint(f0bin + i*f0bin)
// (numpy's arange fill: start + i*delta, delta = (start+step) - start = f0bin exactly), re-centred
// on the measured first harmonic f1 when f1 > fmin and the corrected bin is below M-1 (:464-468)
__device__ __forceinline__ int harmonic_bin(int64_t i, double f0bin, double f1, bool corr, double sr, int M) {
  int nbin = (int)rint(__dadd_rn(f0bin, __dmul_rn((double)i, f0bin)));
  if (i > 0 && corr) {
    const double corrbin = __dmul_rn(__dmul_rn(__ddiv_rn(f1, sr), (double)(2 * M)), (double)(i + 1));
    if (corrbin < (double)(M - 1)) nbin = (int)rint(corrbin);
  }
  return nbin;
}

template <int LOGM>
__global__ void __launch_bounds__(Plan<LOGM>::T) harmonic_kernel(HParams prm) {
  using P = Plan<LOGM>;
  using S = Smem<LOGM>;
  constexpr int M = P::M, T = P::T, NW = P::NW;
  PVK_SMEM(smem);
  constexpr int BUF_STRIDE = S::OFF_BUF1 - S::OFF_BUF0;
  float *famp = reinterpret_cast<float *>(smem + S::OFF_FAMP);
  double *redd = reinterpret_cast<double *>(smem + S::OFF_RED);      // 8 doubles
  double *redc = reinterpret_cast<double *>(smem + S::OFF_HIST);     // 8 doubles (histogram area is free here)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t r0 = (int64_t)blockIdx.x * prm.run;
  const int64_t r1 = (r0 + prm.run < prm.nframes) ? r0 + prm.run : prm.nframes;
  const float2 *twp = prm.tables;
  const float2 *twr = prm.tables + P::TW_TOTAL;
  const int K = prm.npks;
  const double inv_2pidt = 1.0 / (prm.dt * 6.283185307179586), inv_dt = 1.0 / prm.dt;
  int cb = 0;                                                 // PVK_BUF(cb) = spectrum of the last processed frame
  {
    int64_t p = r0 - 1;
    while (p >= 0 && !f0_valid(__ldg(prm.f0 + p))) --p;       // uniform across the CTA
    float2 *pb = PVK_BUF(cb);
    if (p < 0) {
      for (int i = tid; i < P::MP; i += T) pb[i] = make_float2(0.f, 0.f);   // oldfft = zeros (:121)
    } else {
      fft_frame<LOGM>(prm.x + p * (int64_t)prm.hop, prm.win, twp, pb);
      double dummy = 0.0;
      untangle_power<LOGM>(pb, famp, twr, false, dummy);
    }
    __syncthreads();
  }
  for (int64_t r = r0; r < r1; ++r) {
    const int64_t ob = r * K;
    const double thisf = __ldg(prm.f0 + r);
    if (!f0_valid(thisf)) {                                   // skipped frame: zero row, NaN residual (:501-507)
      for (int p = tid; p < K; p += T) { prm.f[ob + p] = 0.0; prm.mag[ob + p] = 0.0; prm.ph[ob + p] = 0.0; }
      if (tid == 0) { prm.residual[r] = __longlong_as_double(0x7ff8000000000000LL); prm.nharm[r] = 0; }
      continue;
    }
    float2 *cur = PVK_BUF(cb ^ 1);
    const float2 *prev = PVK_BUF(cb);
    fft_frame<LOGM>(prm.x + r * (int64_t)prm.hop, prm.win, twp, cur);
    double lsum = 0.0;
    untangle_power<LOGM>(cur, famp, twr, true, lsum);
    {
      const double wsum = warp_sum(lsum);
      if (lane == 0) redd[warp] = wsum;
    }
    __syncthreads();
    double sumsq = redd[0];
#pragma unroll
    for (int w = 1; w < NW; ++w) sumsq += redd[w];
    // harmonics: H = len(np.arange(f0bin, M-1, f0bin)) = ceil((M-1 - f0bin)/f0bin)
    const double f0bin = __dmul_rn(__ddiv_rn(thisf, prm.sr), (double)(2 * M));     // :461
    const double hq = ceil(__ddiv_rn(__dsub_rn((double)(M - 1), f0bin), f0bin));
    const int64_t H = (hq > 0.0 && hq < 4.0e9) ? (int64_t)hq : 0;                   // non-finite f0bin: no harmonics
    double f1 = 0.0;
    bool corr = false;
    if (H > 0) {
      // every thread evaluates the first harmonic itself (identical result, no broadcast)
      double ph0, df0;
      peak_phase_freq(harmonic_bin(0, f0bin, 0.0, false, prm.sr, M), cur, prev, prm.fbin, prm.wfbin, prm.dt, inv_2pidt,
                      inv_dt, ph0, f1, df0);
      corr = f1 > prm.fmin;                                   // :465 (false for NaN)
    }
    double csum = 0.0;
    for (int64_t i = tid; i < H; i += T) {
      const int k = harmonic_bin(i, f0bin, f1, corr, prm.sr, M);
      double thisph, bf, bdf;
      peak_phase_freq(k, cur, prev, prm.fbin, prm.wfbin, prm.dt, inv_2pidt, inv_dt, thisph, bf, bdf);
      // thismagsq = sum(famp[max(k-1,1) : min(k+1,len)+1]**2), left to right (:479-481)
      const int lo = k - 1 > 1 ? k - 1 : 1, hi = k + 1 < M - 1 ? k + 1 : M - 1;
      double s = 0.0;
      for (int m = lo; m <= hi; ++m) s = s + (double)famp[FA(m)];
      csum += s;
      if (i < K) { prm.f[ob + i] = bf; prm.mag[ob + i] = sqrt(s); prm.ph[ob + i] = thisph; }
    }
    for (int64_t p = (H < K ? H : K) + tid; p < K; p += T) { prm.f[ob + p] = 0.0; prm.mag[ob + p] = 0.0; prm.ph[ob + p] = 0.0; }
    {
      const double wc = warp_sum(csum);
      if (lane == 0) redc[warp] = wc;
    }
    __syncthreads();
    if (tid == 0) {
      double cum = redc[0];
      for (int w = 1; w < NW; ++w) cum += redc[w];
      prm.residual[r] = sqrt(sumsq - cum);                    // :490 (NaN when the windows overlap enough)
      prm.nharm[r] = (int32_t)(H < 2147483647 ? H : 2147483647);
    }
    cb ^= 1;                                                  // :491
    __syncthreads();
  }
}

template <int LOGM> static int launch_harmonic(HParams prm, int run_frames, void *stream) {
  using P = Plan<LOGM>;
  const int smem = Smem<LOGM>::bytes(8);
  if (smem > 48 * 1024) {
    if (PVK_SET_SMEM(harmonic_kernel<LOGM>, smem) != 0) {
      set_error("pvk_harmonic: cannot reserve %d bytes of shared memory", smem);
      return PVK_ERR_CUDA;
    }
  }
  int64_t run = run_frames;
  if (run <= 0) {
    run = (prm.nframes + 148 * 7 - 1) / (148 * 7);
    if (run < 8) run = 8;
    if (run > 256) run = 256;
  }
  if (run > prm.nframes) run = prm.nframes;
  prm.run = (int)run;
  const int64_t nblk = (prm.nframes + run - 1) / run;
  PVK_REQUIRE(nblk < (int64_t)2147483647, "pvk_harmonic: grid too large (%lld CTAs)", (long long)nblk);
  PVK_LAUNCH(harmonic_kernel<LOGM>, dim3((unsigned)nblk), dim3(P::T), smem, stream, prm);
  PVK_CHECK_LAUNCH("pvk_harmonic");
  return PVK_OK;
}

// ------------------------------------------------------------------ frame-wise spectral consumers
// FFTFilters.FilterBank.specout (FFTFilters.py:274-292), SoundUtils.RMSWind (SoundUtils.py:74-103)
// and SoundUtils.SpecFlux (:196-231) on the same framing + window + FFT front end as
// analyze_kernel.  One CTA walks a run of frames; the power spectrum |X|^2 of bins 0..M (M =
// nfft/2, Nyquist included) lives in shared memory and every requested output is reduced from it:
//   bank[r, i] = sum_h |X_h|^2 * fbw[i, h]   fbw = the filter folded onto the half spectrum
//                (|X_{N-h}| = |X_h| for a real frame), summed over its support [lo_i, hi_i)
//   rms[r]     = sqrt(sum_n (x_n w_n)^2 / wsum2) through Parseval
//   flux[r-1]  = sqrt(sum_h mult_h (|X_h(r)| - |X_h(r-1)|)^2), mult_h = how many of the bins
//                h, N-h fall in [minbin, maxbin)
struct BParams {
  const float *x;
  const float *win;
  const float2 *tables;
  int hop;
  int64_t nframes;
  int run;
  const double *fbw;
  const int32_t *fb_lo, *fb_hi;
  int nfilt;
  double *bank;
  int minbin, maxbin;
  double *flux;
  double inv_wsum2;
  double *rms;
};

// untangle the packed FFT in `buf` into the power spectrum pw[0..M] (fp32, no FMA contraction:
// bit-identical to numpy float32 re*re + im*im)
template <int LOGM> __device__ __forceinline__ void untangle_to_power(const float2 *buf, float *pw, const float2 *__restrict__ twr) {
  using P = Plan<LOGM>;
  constexpr int M = P::M, T = P::T;
  for (int k = threadIdx.x; k <= M / 2; k += T) {
    if (k == 0) {
      const float2 z0 = buf[PADC(0)];
      const float dc = z0.x + z0.y, ny = z0.x - z0.y;
      pw[0] = __fmul_rn(dc, dc);
      pw[M] = __fmul_rn(ny, ny);
    } else if (k == M / 2) {
      const float2 zh = buf[PADC(M / 2)];
      pw[M / 2] = __fadd_rn(__fmul_rn(zh.x, zh.x), __fmul_rn(zh.y, zh.y));
    } else {
      const float2 a = buf[PADC(k)], bq = buf[PADC(M - k)];
      const float2 e = make_float2(0.5f * (a.x + bq.x), 0.5f * (a.y - bq.y));
      const float2 o = make_float2(0.5f * (a.y + bq.y), -0.5f * (a.x - bq.x));
      const float2 wo = cmul(o, __ldg(twr + k));
      const float2 xa = make_float2(e.x + wo.x, e.y + wo.y);
      const float2 xb = make_float2(e.x - wo.x, -(e.y - wo.y));
      pw[k] = __fadd_rn(__fmul_rn(xa.x, xa.x), __fmul_rn(xa.y, xa.y));
      pw[M - k] = __fadd_rn(__fmul_rn(xb.x, xb.x), __fmul_rn(xb.y, xb.y));
    }
  }
}

template <int LOGM>
__global__ void __launch_bounds__(Plan<LOGM>::T) bank_kernel(BParams prm) {
  using P = Plan<LOGM>;
  using S = Smem<LOGM>;
  constexpr int M = P::M, T = P::T, NW = P::NW, N = 2 * M;
  PVK_SMEM(smem);
  float2 *buf = reinterpret_cast<float2 *>(smem + S::OFF_BUF0);
  float *pws[2] = {reinterpret_cast<float *>(smem + S::OFF_BUF1), reinterpret_cast<float *>(smem + S::OFF_BUF1) + (M + 2)};
  double *redd = reinterpret_cast<double *>(smem + S::OFF_RED);       // 8 doubles
  double *redf = reinterpret_cast<double *>(smem + S::OFF_HIST);      // 8 doubles
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t r0 = (int64_t)blockIdx.x * prm.run;
  const int64_t r1 = (r0 + prm.run < prm.nframes) ? r0 + prm.run : prm.nframes;
  const float2 *twp = prm.tables;
  const float2 *twr = prm.tables + P::TW_TOTAL;
  const bool want_flux = prm.flux != nullptr;
  int cb = 0;
  if (want_flux && r0 > 0) {                                  // spectrum of the frame before the run
    fft_frame<LOGM>(prm.x + (r0 - 1) * (int64_t)prm.hop, prm.win, twp, buf);
    untangle_to_power<LOGM>(buf, pws[cb ^ 1], twr);
    __syncthreads();
  }
  for (int64_t r = r0; r < r1; ++r) {
    float *pw = pws[cb];
    const float *pprev = pws[cb ^ 1];
    fft_frame<LOGM>(prm.x + r * (int64_t)prm.hop, prm.win, twp, buf);
    untangle_to_power<LOGM>(buf, pw, twr);
    __syncthreads();
    if (prm.bank) {                                           // one warp per filter
      for (int i = warp; i < prm.nfilt; i += NW) {
        const int lo = __ldg(prm.fb_lo + i), hi = __ldg(prm.fb_hi + i);
        const double *w = prm.fbw + (int64_t)i * (M + 1);
        double acc = 0.0;
        for (int h = lo + lane; h < hi; h += 32) acc = fma((double)pw[h], __ldg(w + h), acc);
        acc = warp_sum(acc);
        if (lane == 0) prm.bank[r * prm.nfilt + i] = acc;
      }
    }
    if (prm.rms || (want_flux && r > 0)) {
      double e = 0.0, d = 0.0;
      for (int h = tid; h <= M; h += T) {
        const float p = pw[h];
        e += (h == 0 || h == M) ? (double)p : 2.0 * (double)p;
        if (want_flux && r > 0) {
          const int mult = ((h >= prm.minbin && h < prm.maxbin) ? 1 : 0) +
                           ((h != 0 && h != M && N - h >= prm.minbin && N - h < prm.maxbin) ? 1 : 0);
          if (mult) {
            const double df = sqrt((double)p) - sqrt((double)pprev[h]);
            d = fma((double)mult * df, df, d);
          }
        }
      }
      e = warp_sum(e);
      d = warp_sum(d);
      if (lane == 0) { redd[warp] = e; redf[warp] = d; }
      __syncthreads();
      if (tid == 0) {
        double es = redd[0], ds = redf[0];
        for (int w = 1; w < NW; ++w) { es += redd[w]; ds += redf[w]; }
        if (prm.rms) prm.rms[r] = sqrt(es / (double)N * prm.inv_wsum2);
        if (want_flux && r > 0) prm.flux[r - 1] = sqrt(ds);
      }
    }
    if (want_flux) cb ^= 1;
    __syncthreads();
  }
}

template <int LOGM> static int launch_bank(BParams prm, int run_frames, void *stream) {
  using P = Plan<LOGM>;
  const int smem = Smem<LOGM>::bytes(8);
  if (smem > 48 * 1024) {
    if (PVK_SET_SMEM(bank_kernel<LOGM>, smem) != 0) {
      set_error("pvk_stft_bank: cannot reserve %d bytes of shared memory", smem);
      return PVK_ERR_CUDA;
    }
  }
  int64_t run = run_frames;
  if (run <= 0) {
    run = (prm.nframes + 148 * 7 - 1) / (148 * 7);
    if (run < 8) run = 8;
    if (run > 256) run = 256;
  }
  if (run > prm.nframes) run = prm.nframes;
  prm.run = (int)run;
  const int64_t nblk = (prm.nframes + run - 1) / run;
  PVK_REQUIRE(nblk < (int64_t)2147483647, "pvk_stft_bank: grid too large (%lld CTAs)", (long long)nblk);
  PVK_LAUNCH(bank_kernel<LOGM>, dim3((unsigned)nblk), dim3(P::T), smem, stream, prm);
  PVK_CHECK_LAUNCH("pvk_stft_bank");
  return PVK_OK;
}

// ------------------------------------------------------------------ per-frame consumers
// PV.calc_f0 (PVAnalysis.py:371-391) and PV.partial_sum_magnitude (:411-413) over the peak
// table: one warp per frame.
__global__ void frame_stats_kernel(const double *__restrict__ f, const double *__restrict__ mag, int64_t nrows, int K,
                                   double flo, double fhi, double thr, double *__restrict__ fm,
                                   int32_t *__restrict__ fidx, double *__restrict__ psum) {
  const int lane = threadIdx.x & 31;
  const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t row = w0; row < nrows; row += nw) {
    const double *fr = f + row * K, *mr = mag + row * K;
    double mx = __longlong_as_double(0xfff0000000000000LL), sq = 0.0;   // -inf
    for (int c = lane; c < K; c += 32) { const double m = mr[c]; mx = fmax(mx, m); sq += m * m; }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) { mx = fmax(mx, __shfl_xor_sync(FULL, mx, o)); sq += __shfl_xor_sync(FULL, sq, o); }
    const double lim = __dmul_rn(mx, thr);
    // lowest frequency among (f > fmin, f < fmax, mag > max*thr); first column on ties (np.argmin)
    double bf = __longlong_as_double(0x7ff0000000000000LL);   // +inf
    int bc = 0x7fffffff;
    for (int c = lane; c < K; c += 32) {
      const double fv = fr[c];
      if (fv > flo && fv < fhi && mr[c] > lim && (fv < bf || (fv == bf && c < bc))) { bf = fv; bc = c; }
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
      const double of = __shfl_xor_sync(FULL, bf, o);
      const int oc = __shfl_xor_sync(FULL, bc, o);
      if (oc != 0x7fffffff && (bc == 0x7fffffff || of < bf || (of == bf && oc < bc))) { bf = of; bc = oc; }
    }
    if (lane == 0) {
      const bool has = bc != 0x7fffffff;
      fm[row] = has ? bf : 0.0;
      fidx[row] = has ? bc : 0;
      psum[row] = sqrt(sq);
    }
  }
}

// PV.calc_harmonic_power (PVAnalysis.py:266-297), including what :278 really computes: the
// reference indexes ROWS of mag with the column indices of the frame's valid peaks
// (`self.mag[valid_idx]`), so the "magnitudes" summed for a harmonic at column c are the whole
// frame row c of the mag table:  hpower[j, i] = sum over valid h with
// |f_h / round(f_h/f_i) / f_i - 1| < thr  of  rowpow[col_h],  rowpow[c] = sum_k mag[c, k]^2.
// A valid peak in a column >= nrows is an IndexError there; here it raises `*err`.
__global__ void row_power_kernel(const double *__restrict__ mag, int64_t nrows, int K, double *__restrict__ rowpow) {
  const int lane = threadIdx.x & 31;
  const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t row = w0; row < nrows; row += nw) {
    double sq = 0.0;
    for (int c = lane; c < K; c += 32) { const double m = mag[row * K + c]; sq += m * m; }
    sq = warp_sum(sq);
    if (lane == 0) rowpow[row] = sq;
  }
}

__global__ void harmonic_power_kernel(const double *__restrict__ f, const double *__restrict__ rowpow, int64_t nrows, int K,
                                      double thr, double *__restrict__ hpower, double *__restrict__ nharm,
                                      int32_t *__restrict__ err) {
  const int lane = threadIdx.x & 31;
  const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t row = w0; row < nrows; row += nw) {
    const double *fr = f + row * K;
    for (int i = 0; i < K; ++i) {
      const double fi = fr[i];
      double s = 0.0;
      int n = 0;
      if (fi > 0.0) {
        for (int h = lane; h < K; h += 32) {
          const double fh = fr[h];
          if (fh > 0.0) {
            if (h >= nrows) *err = 1;                              // `self.mag[valid_idx]` (:278) is out of range
            double nb = rint(__ddiv_rn(fh, fi));                   // np.round: half to even
            if (nb == 0.0) nb = 1.0;
            const double inh = fabs(__dsub_rn(__ddiv_rn(__ddiv_rn(fh, nb), fi), 1.0));
            if (inh < thr) {
              if (h < nrows) s += rowpow[h];
              ++n;
            }
          }
        }
        s = warp_sum(s);
        n = warp_sum(n);
      }
      if (lane == 0) { hpower[row * K + i] = s; nharm[row * K + i] = (double)n; }
    }
  }
}

// ------------------------------------------------------------------ twiddle tables
template <int LOGM> __global__ void tables_kernel(float2 *tab) {
  using P = Plan<LOGM>;
  constexpr int M = P::M;
  const int gt = blockIdx.x * blockDim.x + threadIdx.x, gs = gridDim.x * blockDim.x;
  for (int q = 1; q < P::NPASS; ++q) {
    const int R = 1 << P::lr(q), PP = 1 << P::lp(q), off = P::tw_off(q);
    for (int e = gt; e < (R - 1) * PP; e += gs) {
      const int r = e / PP + 1, k = e % PP;
      double s, c;
      sincospi(-2.0 * (double)k * (double)r / (double)(PP * R), &s, &c);
      tab[off + e] = make_float2((float)c, (float)s);
    }
  }
  for (int k = gt; k < M / 2; k += gs) {
    double s, c;
    sincospi(-(double)k / (double)M, &s, &c);   // exp(-2*pi*i*k/N), N = 2M
    tab[P::TW_TOTAL + k] = make_float2((float)c, (float)s);
  }
}

template <int LOGM> static int64_t tables_bytes_t() { return (int64_t)(Plan<LOGM>::TW_TOTAL + Plan<LOGM>::M / 2) * 8; }

template <int LOGM> static int launch_tables(void *tables, void *stream) {
  PVK_LAUNCH(tables_kernel<LOGM>, dim3(8), dim3(128), 0, stream, reinterpret_cast<float2 *>(tables));
  PVK_CHECK_LAUNCH("pvk_analyze_init");
  return PVK_OK;
}

// CTAs of `kernel` (block of `threads`, `smem` bytes) the current device holds at once (occupancy x SM count)
template <class Kernel> static int64_t resident_ctas(Kernel kernel, int threads, int smem) {
#ifdef PVK_EMU
  (void)kernel; (void)threads; (void)smem;
  return 148 * 7;
#else
  int dev = 0, sms = 148, occ = 1;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, (size_t)smem) != cudaSuccess || occ < 1) {
    cudaGetLastError();
    occ = 1;
  }
  return (int64_t)sms * occ;
#endif
}

// nfft 1024 / 2048 run analyze_warp_kernel (one warp per frame, AW frames per CTA), every other size
// analyze_kernel (one CTA per frame)
template <int LOGM> static int launch_analyze(AParams prm, int64_t nclips, int run_frames, void *stream) {
  constexpr bool warp_kernel = LOGM == 9 || LOGM == 10;
  auto kernel = [] {
    if constexpr (warp_kernel) return analyze_warp_kernel<LOGM>;
    else return analyze_kernel<LOGM>;
  }();
  constexpr int threads = warp_kernel ? AW * 32 : Plan<LOGM>::T;
  int smem;
  if constexpr (warp_kernel) smem = WSmem<LOGM>::BYTES;
  else smem = Smem<LOGM>::bytes(prm.npks);
  if (smem > 48 * 1024) {
    if (PVK_SET_SMEM(kernel, smem) != 0) {
      set_error("pvk_analyze: cannot reserve %d bytes of shared memory", smem);
      return PVK_ERR_CUDA;
    }
  }
  int64_t run = run_frames;
  if (run <= 0) {
    // The kernel is latency bound (one CTA = one chain of dependent frames, or of groups of AW
    // frames), so what matters is that every resident CTA slot is busy for the same time: size the
    // runs so that the grid is a whole number of waves, as few as possible (every run pays one
    // warm-up frame), with runs of 4..256 frames.
    // Clip batches: every clip is cut into the same number of equally long runs, as many as keep the
    // grid within those waves (a clip's last run is not a short straggler that opens another wave).
    const int64_t slots = resident_ctas(kernel, threads, smem);
    const int64_t total = nclips * prm.nframes;
    const int64_t waves = (total + slots * 256 - 1) / (slots * 256);
    int64_t per_clip = slots * waves / nclips;                 // runs per clip
    const int64_t min_runs = (prm.nframes + 255) / 256;        // runs of at most 256 frames
    if (per_clip < min_runs) per_clip = min_runs;
    run = (prm.nframes + per_clip - 1) / per_clip;
    if (run < 4) run = 4;
  }
  if (run > prm.nframes) run = prm.nframes;
  prm.run = (int)run;
  prm.nruns = (prm.nframes + run - 1) / run;
  const int64_t nblk = nclips * prm.nruns;
  PVK_REQUIRE(nblk < (int64_t)2147483647, "pvk_analyze: grid too large (%lld CTAs)", (long long)nblk);
  PVK_LAUNCH(kernel, dim3((unsigned)nblk), dim3(threads), smem, stream, prm);
  PVK_CHECK_LAUNCH("pvk_analyze");
  return PVK_OK;
}

static int log2_exact(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return (1 << l) == v ? l : -1;
}

#define PVK_DISPATCH_LOGM(logm, CALL)                                                      \
  switch (logm) {                                                                          \
    case 5: return CALL(5);                                                                \
    case 6: return CALL(6);                                                                \
    case 7: return CALL(7);                                                                \
    case 8: return CALL(8);                                                                \
    case 9: return CALL(9);                                                                \
    case 10: return CALL(10);                                                              \
    case 11: return CALL(11);                                                              \
    case 12: return CALL(12);                                                              \
    default: break;                                                                        \
  }

}  // namespace pvk

using namespace pvk;

extern "C" int64_t pvk_analyze_tables_bytes(int nfft) {
  const int l = log2_exact(nfft);
  if (l < 0 || nfft < PVK_MIN_NFFT || nfft > PVK_MAX_NFFT) return -1;
#define CALL(L) tables_bytes_t<L>()
  PVK_DISPATCH_LOGM(l - 1, CALL)
#undef CALL
  return -1;
}

extern "C" int pvk_analyze_init(int nfft, void *tables, void *stream) {
  const int l = log2_exact(nfft);
  PVK_REQUIRE(l >= 0 && nfft >= PVK_MIN_NFFT && nfft <= PVK_MAX_NFFT,
              "pvk_analyze_init: nfft=%d must be a power of two in [%d, %d]", nfft, PVK_MIN_NFFT, PVK_MAX_NFFT);
  PVK_REQUIRE(tables != nullptr, "pvk_analyze_init: tables is NULL");
#define CALL(L) launch_tables<L>(tables, stream)
  PVK_DISPATCH_LOGM(l - 1, CALL)
#undef CALL
  return PVK_ERR_ARG;
}

extern "C" int pvk_analyze_batch(const float *x, int64_t nclips, int64_t clip_stride, int64_t nsamp,
                                 const float *win_scaled, const double *fbin, const double *wfbin,
                                 const void *tables, int nfft, int hop, int npks, double pkthresh,
                                 double dt, double fstep, int64_t frame0, int64_t nframes, int prev_zero,
                                 int run_frames, double *f, double *mag, double *ph, double *realph,
                                 double *binno, int32_t *npk, double *totalmag, float *spec_out,
                                 double *fine_pos, double *fine_val, int64_t out_rows_per_clip, void *stream) {
  PVK_REQUIRE(out_rows_per_clip >= nframes, "pvk_analyze_batch: out_rows_per_clip=%lld < nframes=%lld",
              (long long)out_rows_per_clip, (long long)nframes);
  PVK_REQUIRE(spec_out == nullptr || out_rows_per_clip == nframes,
              "pvk_analyze_batch: spec_out needs out_rows_per_clip=%lld == nframes=%lld (no guard rows)",
              (long long)out_rows_per_clip, (long long)nframes);
  const int l = log2_exact(nfft);
  PVK_REQUIRE(l >= 0 && nfft >= PVK_MIN_NFFT && nfft <= PVK_MAX_NFFT,
              "pvk_analyze: nfft=%d must be a power of two in [%d, %d]", nfft, PVK_MIN_NFFT, PVK_MAX_NFFT);
  PVK_REQUIRE(hop >= 1, "pvk_analyze: hop=%d must be >= 1", hop);
  PVK_REQUIRE(npks >= 1 && npks <= PVK_MAX_NPKS, "pvk_analyze: npks=%d must be in [1, %d]", npks, PVK_MAX_NPKS);
  PVK_REQUIRE(nclips >= 0 && nframes >= 0, "pvk_analyze: negative sizes");
  PVK_REQUIRE(frame0 >= 0 && (prev_zero || frame0 >= 1),
              "pvk_analyze: frame0=%lld needs a warm-up frame (frame0 >= 1) unless prev_zero", (long long)frame0);
  if (nclips == 0 || nframes == 0) return PVK_OK;
  PVK_REQUIRE((frame0 + nframes - 1) * (int64_t)hop + nfft <= nsamp,
              "pvk_analyze: last frame ends at sample %lld > nsamp=%lld",
              (long long)((frame0 + nframes - 1) * (int64_t)hop + nfft), (long long)nsamp);
  PVK_REQUIRE(x && win_scaled && fbin && wfbin && tables && f && mag && ph && realph && binno && npk && totalmag,
              "pvk_analyze: NULL pointer argument");
  PVK_REQUIRE((reinterpret_cast<uintptr_t>(win_scaled) & 7) == 0, "pvk_analyze: win_scaled must be 8-byte aligned");
  AParams prm;
  prm.x = x; prm.clip_stride = clip_stride; prm.win = win_scaled;
  prm.tables = reinterpret_cast<const float2 *>(tables);
  prm.fbin = fbin; prm.wfbin = wfbin; prm.hop = hop; prm.npks = npks;
  prm.pkthresh = pkthresh; prm.dt = dt; prm.fstep = fstep;
  prm.frame0 = frame0; prm.nframes = nframes; prm.prev_zero = prev_zero ? 1 : 0;
  prm.out_rows = out_rows_per_clip;
  prm.run = 0; prm.nruns = 0;                              // chosen by launch_analyze
  prm.f = f; prm.mag = mag; prm.ph = ph; prm.realph = realph; prm.binno = binno;
  prm.npk = npk; prm.totalmag = totalmag;
  prm.spec_out = reinterpret_cast<float2 *>(spec_out);
  PVK_REQUIRE((fine_pos == nullptr) == (fine_val == nullptr), "pvk_analyze: fine_pos and fine_val go together");
  prm.fine_pos = fine_pos; prm.fine_val = fine_val;
#define CALL(L) launch_analyze<L>(prm, nclips, run_frames, stream)
  PVK_DISPATCH_LOGM(l - 1, CALL)
#undef CALL
  return PVK_ERR_ARG;
}

extern "C" int pvk_analyze_ex(const float *x, int64_t nclips, int64_t clip_stride, int64_t nsamp,
                              const float *win_scaled, const double *fbin, const double *wfbin,
                              const void *tables, int nfft, int hop, int npks, double pkthresh,
                              double dt, double fstep, int64_t frame0, int64_t nframes, int prev_zero,
                              int run_frames, double *f, double *mag, double *ph, double *realph,
                              double *binno, int32_t *npk, double *totalmag, float *spec_out,
                              double *fine_pos, double *fine_val, void *stream) {
  return pvk_analyze_batch(x, nclips, clip_stride, nsamp, win_scaled, fbin, wfbin, tables, nfft, hop, npks, pkthresh,
                           dt, fstep, frame0, nframes, prev_zero, run_frames, f, mag, ph, realph, binno, npk, totalmag,
                           spec_out, fine_pos, fine_val, nframes, stream);
}

extern "C" int pvk_analyze(const float *x, int64_t nclips, int64_t clip_stride, int64_t nsamp,
                           const float *win_scaled, const double *fbin, const double *wfbin,
                           const void *tables, int nfft, int hop, int npks, double pkthresh,
                           double dt, double fstep, int64_t frame0, int64_t nframes, int prev_zero,
                           int run_frames, double *f, double *mag, double *ph, double *realph,
                           double *binno, int32_t *npk, double *totalmag, float *spec_out,
                           void *stream) {
  return pvk_analyze_ex(x, nclips, clip_stride, nsamp, win_scaled, fbin, wfbin, tables, nfft, hop, npks, pkthresh,
                        dt, fstep, frame0, nframes, prev_zero, run_frames, f, mag, ph, realph, binno, npk, totalmag,
                        spec_out, nullptr, nullptr, stream);
}

extern "C" int pvk_harmonic(const float *x, int64_t nsamp, const float *win_scaled, const double *fbin,
                            const double *wfbin, const void *tables, int nfft, int hop, int npks, double dt,
                            double sr, double fmin, const double *f0, int64_t nframes, int run_frames,
                            double *f, double *mag, double *ph, double *residual, int32_t *nharm, void *stream) {
  const int l = log2_exact(nfft);
  PVK_REQUIRE(l >= 0 && nfft >= PVK_MIN_NFFT && nfft <= PVK_MAX_NFFT,
              "pvk_harmonic: nfft=%d must be a power of two in [%d, %d]", nfft, PVK_MIN_NFFT, PVK_MAX_NFFT);
  PVK_REQUIRE(hop >= 1, "pvk_harmonic: hop=%d must be >= 1", hop);
  PVK_REQUIRE(npks >= 1 && npks <= PVK_MAX_NPKS, "pvk_harmonic: npks=%d must be in [1, %d]", npks, PVK_MAX_NPKS);
  PVK_REQUIRE(nframes >= 0, "pvk_harmonic: negative sizes");
  if (nframes == 0) return PVK_OK;
  PVK_REQUIRE((nframes - 1) * (int64_t)hop + nfft <= nsamp, "pvk_harmonic: last frame ends at sample %lld > nsamp=%lld",
              (long long)((nframes - 1) * (int64_t)hop + nfft), (long long)nsamp);
  PVK_REQUIRE(x && win_scaled && fbin && wfbin && tables && f0 && f && mag && ph && residual && nharm,
              "pvk_harmonic: NULL pointer argument");
  PVK_REQUIRE((reinterpret_cast<uintptr_t>(win_scaled) & 7) == 0, "pvk_harmonic: win_scaled must be 8-byte aligned");
  HParams prm;
  prm.x = x; prm.win = win_scaled; prm.tables = reinterpret_cast<const float2 *>(tables);
  prm.fbin = fbin; prm.wfbin = wfbin; prm.f0 = f0; prm.hop = hop; prm.npks = npks;
  prm.dt = dt; prm.sr = sr; prm.fmin = fmin; prm.nframes = nframes; prm.run = 0;
  prm.f = f; prm.mag = mag; prm.ph = ph; prm.residual = residual; prm.nharm = nharm;
#define CALL(L) launch_harmonic<L>(prm, run_frames, stream)
  PVK_DISPATCH_LOGM(l - 1, CALL)
#undef CALL
  return PVK_ERR_ARG;
}

extern "C" int pvk_stft_bank(const float *x, int64_t nsamp, const float *win, const void *tables, int nfft, int hop,
                             int64_t nframes, int run_frames, const double *fb_folded, const int32_t *fb_lo,
                             const int32_t *fb_hi, int nfilt, double *bank, int flux_minbin, int flux_maxbin,
                             double *flux, double inv_wsum2, double *rms, void *stream) {
  const int l = log2_exact(nfft);
  PVK_REQUIRE(l >= 0 && nfft >= PVK_MIN_NFFT && nfft <= PVK_MAX_NFFT,
              "pvk_stft_bank: nfft=%d must be a power of two in [%d, %d]", nfft, PVK_MIN_NFFT, PVK_MAX_NFFT);
  PVK_REQUIRE(hop >= 1, "pvk_stft_bank: hop=%d must be >= 1", hop);
  PVK_REQUIRE(nframes >= 0 && nfilt >= 0, "pvk_stft_bank: negative sizes");
  if (nframes == 0) return PVK_OK;
  PVK_REQUIRE((nframes - 1) * (int64_t)hop + nfft <= nsamp, "pvk_stft_bank: last frame ends at sample %lld > nsamp=%lld",
              (long long)((nframes - 1) * (int64_t)hop + nfft), (long long)nsamp);
  PVK_REQUIRE(x && win && tables, "pvk_stft_bank: NULL pointer argument");
  PVK_REQUIRE((reinterpret_cast<uintptr_t>(win) & 7) == 0, "pvk_stft_bank: win must be 8-byte aligned");
  PVK_REQUIRE(bank == nullptr || (nfilt >= 1 && fb_folded && fb_lo && fb_hi),
              "pvk_stft_bank: bank output needs nfilt >= 1 and the folded filter matrix with its supports");
  PVK_REQUIRE(flux == nullptr || (flux_minbin >= 0 && flux_maxbin <= nfft),
              "pvk_stft_bank: flux bins [%d, %d) must lie in [0, nfft]", flux_minbin, flux_maxbin);
  PVK_REQUIRE(bank || flux || rms, "pvk_stft_bank: no output requested");
  BParams prm;
  prm.x = x; prm.win = win; prm.tables = reinterpret_cast<const float2 *>(tables);
  prm.hop = hop; prm.nframes = nframes; prm.run = 0;
  prm.fbw = fb_folded; prm.fb_lo = fb_lo; prm.fb_hi = fb_hi; prm.nfilt = bank ? nfilt : 0; prm.bank = bank;
  prm.minbin = flux_minbin; prm.maxbin = flux_maxbin; prm.flux = flux;
  prm.inv_wsum2 = inv_wsum2; prm.rms = rms;
#define CALL(L) launch_bank<L>(prm, run_frames, stream)
  PVK_DISPATCH_LOGM(l - 1, CALL)
#undef CALL
  return PVK_ERR_ARG;
}

extern "C" int pvk_frame_stats(const double *f, const double *mag, int64_t nrows, int npks, double fmin, double fmax,
                               double thr, double *fm, int32_t *fundamental_idx, double *partial_sum_mag,
                               void *stream) {
  PVK_REQUIRE(nrows >= 0 && npks >= 1, "pvk_frame_stats: bad sizes");
  if (nrows == 0) return PVK_OK;
  PVK_REQUIRE(f && mag && fm && fundamental_idx && partial_sum_mag, "pvk_frame_stats: NULL pointer argument");
  int64_t g = (nrows + 7) / 8;
  if (g > 148 * 32) g = 148 * 32;
  PVK_LAUNCH(frame_stats_kernel, dim3((unsigned)g), dim3(256), 0, stream, f, mag, nrows, npks, fmin, fmax, thr, fm,
             fundamental_idx, partial_sum_mag);
  PVK_CHECK_LAUNCH("pvk_frame_stats");
  return PVK_OK;
}

extern "C" int pvk_harmonic_power(const double *f, const double *mag, int64_t nrows, int npks, double f_threshold,
                                  double *rowpow, double *hpower, double *nharmonics, int32_t *err, void *stream) {
  using namespace pvk;
  PVK_REQUIRE(nrows >= 0 && npks >= 1, "pvk_harmonic_power: bad sizes");
  if (nrows == 0) return PVK_OK;
  PVK_REQUIRE(f && mag && rowpow && hpower && nharmonics && err, "pvk_harmonic_power: NULL pointer argument");
  const int64_t nr = nrows < npks ? nrows : npks;            // only rows that a column index can name
  int64_t g = (nr + 7) / 8;
  PVK_LAUNCH(row_power_kernel, dim3((unsigned)g), dim3(256), 0, stream, mag, nr, npks, rowpow);
  PVK_CHECK_LAUNCH("pvk_harmonic_power");
  g = (nrows + 7) / 8;
  if (g > 148 * 32) g = 148 * 32;
  PVK_LAUNCH(harmonic_power_kernel, dim3((unsigned)g), dim3(256), 0, stream, f, rowpow, nrows, npks, f_threshold, hpower,
             nharmonics, err);
  PVK_CHECK_LAUNCH("pvk_harmonic_power");
  return PVK_OK;
}
