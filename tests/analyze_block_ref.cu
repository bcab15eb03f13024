// analyze_block_ref.cu -- TEST INFRASTRUCTURE ONLY: analyze_kernel<LOGM> (one CTA per frame) at
// nfft 1024 / 2048, the sizes at which the product runs analyze_warp_kernel instead.  The warp
// kernel is meant to compute every output bit for bit as analyze_kernel does; this library lets the
// tests compare the two.  Built by tests/analyze_block_ref.py, for the SIMT emulator with g++ and
// for sm_100a with nvcc; never loaded by the product.
#include "pvk_abi.cu"
#include "pvk_analyze.cu"

namespace pvk {
template <int LOGM> static int launch_block_ref(AParams prm, int64_t nclips, void *stream) {
  const int smem = Smem<LOGM>::bytes(prm.npks);
  if (smem > 48 * 1024 && PVK_SET_SMEM(analyze_kernel<LOGM>, smem) != 0) {
    set_error("pvkt_analyze_block: cannot reserve %d bytes of shared memory", smem);
    return PVK_ERR_CUDA;
  }
  PVK_LAUNCH(analyze_kernel<LOGM>, dim3((unsigned)(nclips * prm.nruns)), dim3(Plan<LOGM>::T), smem, stream, prm);
  PVK_CHECK_LAUNCH("pvkt_analyze_block");
  return PVK_OK;
}
}  // namespace pvk

// The arguments of pvk_analyze_ex, with run_frames (>= 1) the explicit run length of a CTA.
extern "C" int pvkt_analyze_block(const float *x, int64_t nclips, int64_t clip_stride, int64_t nsamp,
                                  const float *win_scaled, const double *fbin, const double *wfbin,
                                  const void *tables, int nfft, int hop, int npks, double pkthresh,
                                  double dt, double fstep, int64_t frame0, int64_t nframes, int prev_zero,
                                  int run_frames, double *f, double *mag, double *ph, double *realph,
                                  double *binno, int32_t *npk, double *totalmag, float *spec_out,
                                  double *fine_pos, double *fine_val, void *stream) {
  PVK_REQUIRE(nfft == 1024 || nfft == 2048, "pvkt_analyze_block: nfft=%d must be 1024 or 2048", nfft);
  PVK_REQUIRE(run_frames >= 1, "pvkt_analyze_block: run_frames=%d must be >= 1", run_frames);
  PVK_REQUIRE(hop >= 1 && npks >= 1 && npks <= PVK_MAX_NPKS && nclips >= 1 && nframes >= 1 &&
                  (prev_zero || frame0 >= 1) && (frame0 + nframes - 1) * (int64_t)hop + nfft <= nsamp,
              "pvkt_analyze_block: bad sizes");
  PVK_REQUIRE((fine_pos == nullptr) == (fine_val == nullptr), "pvkt_analyze_block: fine_pos and fine_val go together");
  AParams prm{};
  prm.x = x; prm.clip_stride = clip_stride; prm.win = win_scaled;
  prm.tables = reinterpret_cast<const float2 *>(tables);
  prm.fbin = fbin; prm.wfbin = wfbin; prm.hop = hop; prm.npks = npks;
  prm.pkthresh = pkthresh; prm.dt = dt; prm.fstep = fstep;
  prm.frame0 = frame0; prm.nframes = nframes; prm.prev_zero = prev_zero ? 1 : 0;
  prm.out_rows = nframes;
  prm.run = (int)(run_frames < nframes ? run_frames : nframes);
  prm.nruns = (nframes + prm.run - 1) / prm.run;
  prm.f = f; prm.mag = mag; prm.ph = ph; prm.realph = realph; prm.binno = binno;
  prm.npk = npk; prm.totalmag = totalmag;
  prm.spec_out = reinterpret_cast<float2 *>(spec_out);
  prm.fine_pos = fine_pos; prm.fine_val = fine_val;
  return nfft == 1024 ? launch_block_ref<9>(prm, nclips, stream) : launch_block_ref<10>(prm, nclips, stream);
}
