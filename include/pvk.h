/*
 * pvk.h -- C ABI of the B200-native phase-vocoder kernels (libpvk.so).
 *
 * The reference (goiosunsw/PyPeVoc) is pure Python and has no FFI / plugin boundary for
 * this path; its interface is the Python class pypevoc.PV (pypevoc/PVAnalysis.py:71-417)
 * and pypevoc.SinSum (:797-1111).  Every entry point below names the reference method it
 * replaces; pypevoc_b200/pv.py is the Python host side that mirrors those classes and
 * reaches these symbols through ctypes (see INTEGRATION.md for the binding a PyPeVoc
 * maintainer would add).
 *
 * Conventions
 *   - plain pointers and sizes only; all data pointers are DEVICE pointers (cudaMalloc /
 *     torch tensor .data_ptr()) on the current device unless named host_*.
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL =
 *     legacy default stream) and keeps no global state besides a thread-local error
 *     string; re-entrant across streams and devices.
 *   - the library never allocates user-visible memory: outputs and scratch are caller
 *     provided, scratch sizes come from the *_bytes() queries.
 *   - return value 0 = ok; non-zero = error, text in pvk_last_error().  Nothing throws.
 */
#ifndef PVK_H_
#define PVK_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PVK_OK 0
#define PVK_ERR_ARG 1
#define PVK_ERR_CUDA 2

#define PVK_MIN_NFFT 64
#define PVK_MAX_NFFT 8192
#define PVK_MAX_NPKS 1024

/* ABI version (bumped on any signature change). */
int pvk_version(void);

/* Thread-local text of the last error on this thread ("" if none). */
const char *pvk_last_error(void);

/* Number of kernels this library has launched in this process so far (diagnostics / benchmarks). */
int64_t pvk_launch_count(void);

/* ------------------------------------------------------------------ analysis
 * Replaces PV.run_pv / PV.calc_pv_frame / PV.calc_fft_frame / PV.dphase2freq
 * (PVAnalysis.py:133-264) and the PeakFinder calls they make (PeakFinder.py:35-74,
 * 113-134,155-194).
 */

/* Bytes of device scratch pvk_analyze_init() fills with twiddle tables for `nfft`. */
int64_t pvk_analyze_tables_bytes(int nfft);

/* Fill `tables` (pvk_analyze_tables_bytes(nfft) bytes) once per (device, nfft). */
int pvk_analyze_init(int nfft, void *tables, void *stream);

/*
 * Analyse `nframes` frames of each of `nclips` signals.
 *
 *   x            fp32 samples; clip c starts at x + c*clip_stride and holds nsamp samples
 *   win_scaled   nfft floats: wind(nfft) / wfact          (PVAnalysis.py:97-102,157)
 *   fbin, wfbin  nfft doubles each, computed by the host with the reference's own numpy
 *                expressions                              (PVAnalysis.py:114-118)
 *   dt, fstep    hop/sr and sr/nfft                       (PVAnalysis.py:105-108)
 *   pkthresh     PeakFinder minrattomax                   (PVAnalysis.py:175)
 *   frame0       local index of the first frame to emit: output row r is the frame that
 *                starts at sample (frame0 + r)*hop of its clip
 *   prev_zero    1: the frame before `frame0` is the all-zero spectrum PV starts from
 *                (PVAnalysis.py:121); 0: frame0-1 (>= 0) is recomputed as warm-up
 *                (segment sharding, SURVEY 8e)
 *   run_frames   frames one CTA walks through (0 = library default)
 *
 * Outputs, in the reference's own layout (PVAnalysis.py:226-264): float64
 * [nclips, nframes, npks] zero padded f / mag / ph / realph / binno, plus npk int32
 * [nclips, nframes] (valid entries per row) and totalmag float64 [nclips, nframes].
 * spec_out (optional, may be NULL): complex64 [nclips, nframes, nfft/2] =
 * calc_fft_frame(pos)[:nfft/2] (PVAnalysis.py:150-158,169) as (re, im) float pairs.
 */
int pvk_analyze(const float *x, int64_t nclips, int64_t clip_stride, int64_t nsamp,
                const float *win_scaled, const double *fbin, const double *wfbin,
                const void *tables, int nfft, int hop, int npks, double pkthresh,
                double dt, double fstep, int64_t frame0, int64_t nframes, int prev_zero,
                int run_frames, double *f, double *mag, double *ph, double *realph,
                double *binno, int32_t *npk, double *totalmag, float *spec_out,
                void *stream);

/*
 * pvk_analyze with two more optional outputs (both NULL or both set): float64
 * [nclips, nframes, npks] fine_pos / fine_val = PeakFinder.refine (PeakFinder.py:331-372,
 * fun=None, default x) of every emitted peak on famp = |fx|: the vertex of the parabola through
 * the three bins around the peak (position in bins, value).  PV itself never calls refine
 * (PVAnalysis.py:175-178 keeps integer positions): this is the opt-in "quadratic bin
 * interpolation" of the peak kernel, columns aligned with f / mag / binno.
 */
int pvk_analyze_ex(const float *x, int64_t nclips, int64_t clip_stride, int64_t nsamp,
                   const float *win_scaled, const double *fbin, const double *wfbin,
                   const void *tables, int nfft, int hop, int npks, double pkthresh,
                   double dt, double fstep, int64_t frame0, int64_t nframes, int prev_zero,
                   int run_frames, double *f, double *mag, double *ph, double *realph,
                   double *binno, int32_t *npk, double *totalmag, float *spec_out,
                   double *fine_pos, double *fine_val, void *stream);

/*
 * pvk_analyze_ex for clip batches that continue into tracking and resynthesis (BASELINE
 * configs[2]; SURVEY 8b "pvk_analyze_batch", PVAnalysis.py:213-264 once per clip): clip c writes
 * its rows at row index c * out_rows_per_clip + r of every output table, out_rows_per_clip >=
 * nframes.  The rows in between are the caller's guard rows: kept all-zero they end every
 * partial at a clip boundary, so ONE pvk_track / pvk_track_pack / pvk_resynth over the flattened
 * [nclips * out_rows_per_clip, npks] tables links, packs and renders all clips at once, each
 * exactly like a PV of its own (ids are numbered clip after clip).
 * fine_pos / fine_val (optional) follow the same layout, float64 [nclips, out_rows_per_clip,
 * npks]; the kernel writes only the nframes rows of each clip, so the caller zeroes their guard
 * rows as those of the other tables.  spec_out must be NULL unless out_rows_per_clip == nframes
 * (PVK_ERR_ARG otherwise): the spectrum has no guard rows.
 */
int pvk_analyze_batch(const float *x, int64_t nclips, int64_t clip_stride, int64_t nsamp,
                      const float *win_scaled, const double *fbin, const double *wfbin,
                      const void *tables, int nfft, int hop, int npks, double pkthresh,
                      double dt, double fstep, int64_t frame0, int64_t nframes, int prev_zero,
                      int run_frames, double *f, double *mag, double *ph, double *realph,
                      double *binno, int32_t *npk, double *totalmag, float *spec_out,
                      double *fine_pos, double *fine_val, int64_t out_rows_per_clip, void *stream);

/* ------------------------------------------------------------------ f0-guided analysis
 * Replaces PVHarmonic.run_pv / PVHarmonic.calc_pv_frame (PVAnalysis.py:419-538) for one
 * signal: frame r (starting at sample r*hop) is processed when f0[r] > 0 and not NaN (:509);
 * its bins are round(arange(f0bin, nfft/2-1, f0bin)), f0bin = f0[r]/sr*nfft (:461-462), the
 * harmonics above the first re-centred on the measured first harmonic when that exceeds
 * `fmin` (:464-468); per harmonic dphase2freq, the 3-bin magnitude and the phase (:471-488).
 * The phase difference is taken against the last PROCESSED frame (:491), all-zero before the
 * first one (:121).
 *
 *   f0        float64 [nframes]  (what set_f0 leaves in PVHarmonic.f0, :424-441)
 *   f mag ph  float64 [nframes, npks], cut / zero padded to npks (:512-516); skipped frames
 *             are zero rows
 *   residual  float64 [nframes]: sqrt(sum(famp^2) - sum over ALL harmonics of their 3-bin
 *             powers) (:490), NaN for skipped frames (:507)
 *   nharm     int32 [nframes]: number of harmonics evaluated (len(bins)), 0 for skipped frames
 */
int pvk_harmonic(const float *x, int64_t nsamp, const float *win_scaled, const double *fbin,
                 const double *wfbin, const void *tables, int nfft, int hop, int npks, double dt,
                 double sr, double fmin, const double *f0, int64_t nframes, int run_frames,
                 double *f, double *mag, double *ph, double *residual, int32_t *nharm, void *stream);

/* ------------------------------------------------------------------ frame-wise spectral consumers
 * The framing + window + FFT front end of pvk_analyze for the reference's other frame loops:
 * FFTFilters.FilterBank.specout (pypevoc/FFTFilters.py:274-292; mel / MFCC banks :300-374),
 * SoundUtils.RMSWind (pypevoc/SoundUtils.py:74-103) and SoundUtils.SpecFlux (:196-231).
 * Frame r covers samples [r*hop, r*hop + nfft); `win` float32 [nfft] is the raw window.
 * Any of the three outputs may be NULL (at least one is required):
 *   bank  float64 [nframes, nfilt]: sum over ALL nfft bins of |FFT|^2 * fb[i, :] (:285-288), with
 *         the filter folded onto bins 0..nfft/2 by the caller: fb_folded float64
 *         [nfilt, nfft/2 + 1], fb_folded[i, h] = fb[i, h] + fb[i, nfft - h] (0 < h < nfft/2),
 *         and the support of every row as fb_lo / fb_hi int32 [nfilt] (zero weights outside
 *         [lo, hi) are skipped)
 *   flux  float64 [nframes - 1]: flux[j] = sqrt(sum_{k in [minbin, maxbin)} (|X_j[k]| -
 *         |X_{j+1}[k]|)^2) over bins of the full nfft-point spectrum (SoundUtils.py:222-225)
 *   rms   float64 [nframes]: sqrt(sum((x*win)^2) * inv_wsum2) (SoundUtils.py:96,103)
 */
int pvk_stft_bank(const float *x, int64_t nsamp, const float *win, const void *tables, int nfft, int hop,
                  int64_t nframes, int run_frames, const double *fb_folded, const int32_t *fb_lo,
                  const int32_t *fb_hi, int nfilt, double *bank, int flux_minbin, int flux_maxbin,
                  double *flux, double inv_wsum2, double *rms, void *stream);

/* ------------------------------------------------------------------ per-frame consumers
 * PV.calc_f0 (PVAnalysis.py:371-391) and PV.partial_sum_magnitude (:411-413) over peak tables
 * f, mag float64 [nrows, npks]:
 *   fm              float64 [nrows]: lowest frequency with fmin < f < fmax and
 *                   mag > max(mag)*thr (first column on ties), 0 when there is none
 *   fundamental_idx int32 [nrows]: its column (0 when there is none)
 *   partial_sum_mag float64 [nrows]: sqrt(sum(mag^2))
 */
int pvk_frame_stats(const double *f, const double *mag, int64_t nrows, int npks, double fmin, double fmax,
                    double thr, double *fm, int32_t *fundamental_idx, double *partial_sum_mag,
                    void *stream);

/* PV.calc_harmonic_power (PVAnalysis.py:266-297) over peak tables f, mag float64 [nrows, npks]:
 *   hpower, nharmonics float64 [nrows, npks]: for every valid peak i (f > 0) of a frame, the
 *   valid peaks h of the same frame with |f_h / round(f_h / f_i) / f_i - 1| < f_threshold are
 *   counted (nharmonics) and -- exactly as :278 indexes `self.mag[valid_idx]`, i.e. ROWS of the
 *   table by the peaks' COLUMN numbers -- hpower sums rowpow[column of h] over them, where
 *   rowpow[c] = sum_k mag[c, k]^2; 0 in columns without a peak.
 *   rowpow: scratch, float64 [min(nrows, npks)].  err: int32 [1], zeroed by the caller; set to 1
 *   when a harmonic's column number is >= nrows (IndexError in the reference).
 */
int pvk_harmonic_power(const double *f, const double *mag, int64_t nrows, int npks, double f_threshold,
                       double *rowpow, double *hpower, double *nharmonics, int32_t *err, void *stream);

/* ------------------------------------------------------------------ tracking
 * Replaces PV.toSinSum -> SinSum.add_frame (PVAnalysis.py:299-322,871-957).
 *
 * Input: f, mag float64 [nclips, nframes, npks] (rows in the reference layout; a slot is a
 * point iff f > 0 and mag > 0, :876).
 * Output:
 *   link  int32 [nclips, nframes, npks]: column of the continued peak in the previous frame
 *         (>= 0), -1 = not a point, <= -2 = starts a new partial (rank -2-link among the
 *         frame's new partials in processing order, :941)
 *   tid   int32 [nclips, nframes, npks]: track (partial) id per slot, -1 = not a point; ids
 *         numbered per clip in add_empty_partial call order (:819-830), i.e. the index of
 *         the partial in the reference's ss.partial list
 *   ntracks int32 [nclips]: number of partials per clip
 */
int64_t pvk_track_workspace_bytes(int64_t nclips, int64_t nframes, int npks);

int pvk_track(const double *f, const double *mag, int64_t nclips, int64_t nframes, int npks,
              double maxpitchjmp, int32_t *tid, int32_t *link, int32_t *ntracks,
              void *workspace, int64_t workspace_bytes, void *stream);

/* First frame and length of every partial from a track-id table alone (tstart / tlen int32
 * [ntracks] = ss.st and ss.end - ss.st + 1, :827-828,950); ids >= ntracks must not occur.  Used
 * on the gathered global id table of a sharded run. */
int pvk_track_spans(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                    int32_t *tstart, int32_t *tlen, void *stream);

/* Sizes of a track-id table in one small read-back: stats int64 [3][nclips] = number of points
 * (= sum of len(partial.f), the length of the packed arrays of pvk_track_pack) | last frame
 * holding a point (= max(ss.end), :1059; -1 = none) | number of partials (copy of ntracks). */
int pvk_track_stats(const int32_t *tid, const int32_t *ntracks, int64_t nclips, int64_t nframes,
                    int npks, int64_t *stats, void *stream);

/* Clip batches flattened with pvk_analyze_batch (rows_per_clip rows per clip, zero guard rows):
 * from the packed tracks' first frames / lengths, count[c] = partials of clip c (their ids are the
 * exclusive scan of count, clip after clip) and last[c] = last local frame of clip c holding a
 * point (-1: none) = max(SinSum.end) of that clip (PVAnalysis.py:1059).  int32 [nclips] each. */
int pvk_clip_spans(const int32_t *tstart, const int32_t *tlen, int64_t ntracks, int64_t rows_per_clip,
                   int64_t nclips, int32_t *count, int32_t *last, void *stream);

/* Pack per-track value runs (= RegPartial.f/mag/ph/realph lists, :616-626, with
 * start_idx = tstart, :598) from the frame tables of ONE clip.  ntracks is the value
 * pvk_track reported -- or any smaller capacity of the index arrays (a pack launched before the
 * count has been read back): ids >= ntracks are skipped, nothing is written outside
 * tstart/tlen[0..ntracks), toff[0..ntracks] and the first nframes*npks packed slots, and the
 * partials below ntracks come out exactly as in a full pack.  Outputs: tstart / tlen int32 [ntracks] (= ss.st and
 * ss.end - ss.st + 1, :827-828,950), toff int64 [ntracks+1] exclusive offsets, packed
 * float64 arrays of length sum(tlen) (pph may be NULL).  workspace: scratch of
 * pvk_track_pack_workspace_bytes(ntracks) bytes. */
int64_t pvk_track_pack_workspace_bytes(int64_t ntracks);

int pvk_track_pack(const double *f, const double *mag, const double *ph, const double *realph,
                   const int32_t *tid, int64_t nframes, int npks,
                   int64_t ntracks, int32_t *tstart, int32_t *tlen, int64_t *toff, double *pf,
                   double *pmag, double *pph, double *prealph, void *workspace,
                   int64_t workspace_bytes, void *stream);

/* pvk_track_pack sized by an upper bound: `ntracks` is the CAPACITY of tstart / tlen / toff, the
 * real number of partials is read on the device from ntracks_dev[0] (pvk_track's output; NULL =
 * `ntracks` itself).  Lets a caller queue the pack -- and the resynthesis, pvk_resynth_dev --
 * behind the link kernels before it has read any count back: no host round trip in the middle of
 * the hot path.  Entries beyond the real count are left untouched; toff[real count] = number of
 * points. */
int pvk_track_pack_dev(const double *f, const double *mag, const double *ph, const double *realph,
                       const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                       const int32_t *ntracks_dev, int32_t *tstart, int32_t *tlen, int64_t *toff,
                       double *pf, double *pmag, double *pph, double *prealph, void *workspace,
                       int64_t workspace_bytes, void *stream);

/* Renumber a table remapped by any map, in any order (DESIGN.md 4.3, "Remap"): tid_map [nrows_out, npks]
 * holds the SOURCE ids of pvk_time_map's tid_out under the map tmap (nrows_out float64 frames in
 * [0, nframes - 1]), and a source partial read backwards or across a jump covers several runs of
 * consecutive output rows.  Slot (b, c) holding source partial v continues v's run when b > 0 and
 * tstart[v] <= floor(tmap[b - 1]) <= tstart[v] + tlen[v] - 1; otherwise it starts a new run.  Every run
 * becomes one partial, numbered in ascending order of (first output row, source id):
 *   link_out  int32 [nrows_out, npks], pvk_track's encoding: the column of the slot in row b - 1 (>= 0),
 *             -1 = not a point, <= -2 = new run of rank -2 - link among the row's new runs by source id
 *   tid_out   int32 [nrows_out, npks]: run id per slot, -1 = not a point
 *   ntracks_out  int32 [1]: number of runs
 * The result is a valid track table: pvk_track_stats counts it and pvk_track_pack packs it with the
 * tables of pvk_time_map.  With a non-decreasing map it is the time map's table with the partials it
 * skips removed and the ids compacted in order.
 *   tid_src, nframes, ntracks_src, tstart, tlen, toff   the source table [nframes, npks] and its pack
 *   workspace    pvk_track_relink_workspace_bytes(nframes, npks, nrows_out) bytes
 * Checks sizes, npks, pointers and nrows_out * npks < 2^31 before any CUDA call; allocates nothing. */
int64_t pvk_track_relink_workspace_bytes(int64_t nframes, int npks, int64_t nrows_out);

int pvk_track_relink(const int32_t *tid_src, int64_t nframes, int npks, int64_t ntracks_src,
                     const int32_t *tstart, const int32_t *tlen, const int64_t *toff, const int32_t *tid_map,
                     const double *tmap, int64_t nrows_out, int32_t *tid_out, int32_t *link_out,
                     int32_t *ntracks_out, void *workspace, int64_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------ segment sharding
 * A long signal split into per-GPU frame ranges is linked per segment (pvk_track on the
 * segment's window of rows: `own0` halo rows, then `nown` own rows, then more halo rows); these
 * three calls give the own rows the numbering the unsharded pvk_track would give them
 * (partials in order of creation, PVAnalysis.py:819-830).  See pypevoc_b200/dist.py.
 *
 * pvk_segment_summary: int32 summary[2*npks + 4] of one segment = local ids of the row before
 *   the first own row (-1 = none) | local ids of the last own row | partials born before the
 *   own rows | those + partials born in the own rows | global index (j0 + local) of the last own
 *   row holding a point (-1 = none) | nown.  The summaries of all segments are exchanged with
 *   one small all_gather.
 * pvk_segment_resolve: sequential pass over the gathered summaries [world][2*npks + 4] for
 *   segment `rank`: gidlow[v] = global id of local id v for the partials born before the own
 *   rows (v < summary[2K]; gidlow and scratch: at least npks * the largest own0 of any segment ints
 *   each, scratch_ints says how many), params[8] = {global
 *   id of the first partial born in the own rows, partials born before the own rows, partials
 *   born in them, total number of partials, global index of the last frame with a point, ...}.
 * pvk_segment_rename: tid_global[e] for the n = nown*npks slots of the own rows.
 */
int pvk_segment_summary(const int32_t *tid, int npks, int64_t own0, int64_t nown, int64_t j0,
                        int32_t *summary, void *stream);
int pvk_segment_resolve(const int32_t *summaries, int world, int npks, int rank, int32_t *scratch,
                        int64_t scratch_ints, int32_t *gidlow, int32_t *params, void *stream);
int pvk_segment_rename(const int32_t *tid_own, int64_t n, const int32_t *gidlow,
                       const int32_t *params, int32_t *tid_global, void *stream);

/*
 * pvk_segment_rename fused with the gather of the track table (no reference counterpart; replaces
 * pvk_segment_rename + an all_gather): the n renamed ids are stored at element offset `dst_offset`
 * (= first own row * npks) of EVERY table in dst_tables[0..ndst) -- a DEVICE array of device
 * pointers to the int32 [frames_total, npks] tables of all ranks, the remote ones being peer memory
 * mapped over NVLink (CUDA IPC / symmetric memory).  P2P stores from the kernel that computes the
 * ids; the caller provides the cross-rank barriers before (tables free) and after (stores visible).
 */
int pvk_segment_rename_push(const int32_t *tid_own, int64_t n, const int32_t *gidlow, const int32_t *params,
                            int32_t *const *dst_tables, int ndst, int64_t dst_offset, void *stream);

/*
 * pvk_segment_rename_push through NVSwitch multicast: `mc_table` is the MULTICAST address of the
 * ranks' int32 [frames_total, npks] tables (one symmetric allocation of every rank bound to a
 * multicast object).  Every 16 bytes of renamed ids leave this GPU once (multimem.st) and the switch
 * writes them into the table of every rank, this one included.  Barriers as for the push variant.
 */
int pvk_segment_rename_mcast(const int32_t *tid_own, int64_t n, const int32_t *gidlow, const int32_t *params,
                             int32_t *mc_table, int64_t dst_offset, void *stream);

/* ------------------------------------------------------------------ resynthesis
 * Replaces SinSum.synth -> RegPartial.synth (PVAnalysis.py:1053-1070,684-756),
 * phase_preserve=True path, for ONE clip (pvk_resynth_ex below: phase_preserve=False).
 *
 *   tid [nframes, npks]                  track id per frame slot (pvk_track)
 *   ntracks, tstart/tlen/toff, pf/pmag/prealph   the packed partials (pvk_track_pack); partials
 *                                        shorter than minframes are skipped (:1061)
 *   sr, hop      synthesis sample rate and hop (hop may differ from the analysis hop)
 *   nfft, hop_an analysis parameters the SinSum was built with (:824-825,1055)
 *   nout         length of the whole signal, (max_end+2)*hop + int(edge*hop*nfft/hop_an/2)
 *                (:1059,1070)
 *   block0, nblocks  render output blocks [block0, block0+nblocks) of `hop` samples
 *                (multi-GPU: each rank renders a disjoint block range); nblocks < 0 = all
 *   out          float64; out[0] is sample block0*hop; every sample of the rendered block
 *                range below nout is written (zeros where no partial sounds)
 *   workspace    scratch: start / end slot masks and fade parameters of the rendered
 *                partials plus the staged per-block coefficients of one chunk of blocks.
 *                pvk_resynth_workspace_bytes() gives the recommended size (chunks of up to
 *                32768 blocks); any size that holds the fixed part and one block works,
 *                smaller workspaces only mean more, smaller launches.
 *   reuse_tracks 1: the workspace still holds the masks and fade parameters written by an
 *                earlier call with the same partials, hop, nfft, hop_an, edge and minframes
 *                (rendering one signal in several block ranges); 0: compute them
 */
int64_t pvk_resynth_workspace_bytes(int64_t nframes, int npks, int64_t ntracks, int64_t nblocks);

int pvk_resynth(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                const int32_t *tstart, const int32_t *tlen, const int64_t *toff, const double *pf,
                const double *pmag, const double *prealph, double sr, int hop, int nfft,
                int hop_an, double edge, int minframes, double *out, int64_t nout,
                int64_t block0, int64_t nblocks, void *workspace, int64_t workspace_bytes,
                int reuse_tracks, void *stream);

/* pvk_resynth with the number of partials on the device (see pvk_track_pack_dev): `ntracks` is the
 * capacity the workspace was sized for, ntracks_dev[0] the real count (NULL = `ntracks`).  `nout`
 * may then be an upper bound, (nframes + 1) * hop + edge samples: samples beyond the real signal
 * length are rendered into the caller's (larger) buffer and cut by the caller once it has read
 * max(end) back. */
int pvk_resynth_dev(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                    const int32_t *ntracks_dev, const int32_t *tstart, const int32_t *tlen,
                    const int64_t *toff, const double *pf, const double *pmag, const double *prealph,
                    double sr, int hop, int nfft, int hop_an, double edge, int minframes, double *out,
                    int64_t nout, int64_t block0, int64_t nblocks, void *workspace,
                    int64_t workspace_bytes, int reuse_tracks, void *stream);

/* pvk_resynth_dev with a choice of phase model (pvk_resynth_dev = pvk_resynth_ex(..., 1, 1.0, NULL, 0)).
 *   phase_preserve  1: the reference's phase-preserving model above (every block re-anchored at the
 *                   analysed realph); fscale must be 1.
 *                   0: integrated phase -- theta(s) = realph[0] + 2 pi fscale / sr * sum_{m<s} fsig[m]
 *                   over the whole body of a partial, heads / tails at the scaled first / last frequency
 *                   (DESIGN.md 4.3).  A synthesis hop other than the analysis hop stretches time, fscale
 *                   shifts pitch; partials with fscale * max(f) >= sr / 2 are not rendered.
 *   fscale       frequency ratio, finite and > 0
 *   phase_ws     integrated phase only: scratch of one double per packed point (phase_ws_len >=
 *                toff[ntracks]; an upper bound such as nframes * npks when the count is on the device).
 *                Written when reuse_tracks = 0 and read by every call, so calls rendering one signal in
 *                block ranges pass the same buffer.  A length below min(ntracks, nframes * npks) is
 *                rejected; partials whose points lie beyond phase_ws_len are not rendered.
 */
int pvk_resynth_ex(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                   const int32_t *ntracks_dev, const int32_t *tstart, const int32_t *tlen,
                   const int64_t *toff, const double *pf, const double *pmag, const double *prealph,
                   double sr, int hop, int nfft, int hop_an, double edge, int minframes, double *out,
                   int64_t nout, int64_t block0, int64_t nblocks, void *workspace,
                   int64_t workspace_bytes, int reuse_tracks, int phase_preserve, double fscale,
                   double *phase_ws, int64_t phase_ws_len, void *stream);

/* pvk_resynth_ex with phase_preserve = 0, minus the phase scan: the block start phases in phase_ws and
 * the Nyquist flags in the workspace were written by pvk_resynth_scan (+ pvk_resynth_handover /
 * pvk_resynth_import_flags).  reuse_tracks = 0 computes the masks and fades from them; later block
 * ranges of the same signal go through pvk_resynth_ex(reuse_tracks = 1).  phase_preserve must be 0. */
int pvk_resynth_render(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                       const int32_t *ntracks_dev, const int32_t *tstart, const int32_t *tlen,
                       const int64_t *toff, const double *pf, const double *pmag, const double *prealph,
                       double sr, int hop, int nfft, int hop_an, double edge, int minframes, double *out,
                       int64_t nout, int64_t block0, int64_t nblocks, void *workspace,
                       int64_t workspace_bytes, int reuse_tracks, int phase_preserve, double fscale,
                       double *phase_ws, int64_t phase_ws_len, void *stream);

/* ------------------------------------------------------------------ integrated phase of a sharded signal
 * One long signal split over ranks (dist.py): each rank scans the partials of its window rows only.
 * The three calls below carry the true phases and the Nyquist rule across the ranks (DESIGN.md 4.3):
 *
 * pvk_resynth_scan -- the phase scan of pvk_resynth_ex (block start phases into phase_ws, local Nyquist
 *   flags into the workspace), plus, when rec != NULL, this rank's hand-over record for local row h_hi
 *   (the next rank's hand-over row; < 0: none): int64 rec[2 * npks], rec[k] = the column in local row
 *   h_lo of the partial in column k of row h_hi (-1: born after h_lo or h_lo < 0, value absolute; -2: no
 *   partial), rec[npks + k] = P(h_hi) - P(h_lo) or P(h_hi), 63-bit fixed point.  h_lo < 0: the window
 *   starts at frame 0 (nothing cut).
 * pvk_resynth_handover -- composes the records of ranks [0, rank) (recs [world][2 * npks], all ranks'
 *   records as an all_gather leaves them) into the true P at local row h_lo and shifts the partials
 *   alive there.  No-op for h_lo < 0 or rank 0.
 * pvk_nyquist_flags -- flags[gid[i]] = 1 where fscale * f[i] >= sr / 2, over n points (this rank's own
 *   rows and their global ids); the flags of all ranks are then OR-ed (all_reduce MAX).
 * pvk_resynth_import_flags -- the global flags into the workspace: local partial v takes the flag of the
 *   global id table[row0 + tstart[v]] holds in its slot (table [table_rows, npks]: the global track
 *   table, row0: the global row of local row 0).
 * All four check their arguments before any CUDA call.  Workspace: as pvk_resynth_ex's.
 */
int pvk_resynth_scan(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks, const int32_t *tstart,
                     const int32_t *tlen, const int64_t *toff, const double *pf, const double *prealph, double sr,
                     int hop, int nfft, int hop_an, double fscale, void *workspace, int64_t workspace_bytes,
                     double *phase_ws, int64_t phase_ws_len, int64_t h_lo, int64_t h_hi, int64_t *rec,
                     int64_t rec_len, void *stream);
int pvk_resynth_handover(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks, const int32_t *tstart,
                         const int32_t *tlen, const int64_t *toff, double *phase_ws, int64_t phase_ws_len,
                         const int64_t *recs, int64_t recs_len, int world, int rank, int64_t h_lo, void *workspace,
                         int64_t workspace_bytes, void *stream);
int pvk_nyquist_flags(const double *f, const int32_t *gid, int64_t n, double sr, double fscale, uint8_t *flags,
                      int64_t nflags, void *stream);
int pvk_resynth_import_flags(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks, const int32_t *tstart,
                             const int32_t *table, int64_t table_rows, int64_t row0, const uint8_t *flags,
                             int64_t nflags, void *workspace, int64_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------ time-varying frequency ratio
 * The _curve variants take, after fscale, a frequency-ratio curve: fcurve[row] (device, fcurve_len
 * doubles) is the ratio of every partial in frame row `row` of the table, i.e. of output block `row`,
 * in place of fscale (DESIGN.md 4.3).  The block advances, the in-block phase polynomial and the Nyquist
 * test of a point use the ratio of its own row; a head runs at the ratio of its partial's first row, a
 * tail at that of its last row.  The phase stays continuous at every block edge; the frequency steps by
 * fcurve[b + 1] / fcurve[b] there.  fcurve = NULL: exactly the variant without _curve.  A non-NULL
 * fcurve needs fcurve_len >= the number of rows (nframes; n / npks for pvk_nyquist_flags_curve, whose
 * f / gid are whole rows of npks slots), fscale == 1 and phase_preserve == 0; these are checked before
 * any CUDA call.  The values (finite, > 0) are the caller's to check.  A constant curve c renders the
 * same bits as fscale = c.  A sharded rank passes the rows of its window (pvk_nyquist_flags_curve: of
 * its own rows); pvk_resynth_handover needs no curve.
 */
int pvk_resynth_ex_curve(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                         const int32_t *ntracks_dev, const int32_t *tstart, const int32_t *tlen,
                         const int64_t *toff, const double *pf, const double *pmag, const double *prealph,
                         double sr, int hop, int nfft, int hop_an, double edge, int minframes, double *out,
                         int64_t nout, int64_t block0, int64_t nblocks, void *workspace,
                         int64_t workspace_bytes, int reuse_tracks, int phase_preserve, double fscale,
                         const double *fcurve, int64_t fcurve_len, double *phase_ws, int64_t phase_ws_len,
                         void *stream);
int pvk_resynth_render_curve(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks,
                             const int32_t *ntracks_dev, const int32_t *tstart, const int32_t *tlen,
                             const int64_t *toff, const double *pf, const double *pmag, const double *prealph,
                             double sr, int hop, int nfft, int hop_an, double edge, int minframes, double *out,
                             int64_t nout, int64_t block0, int64_t nblocks, void *workspace,
                             int64_t workspace_bytes, int reuse_tracks, int phase_preserve, double fscale,
                             const double *fcurve, int64_t fcurve_len, double *phase_ws, int64_t phase_ws_len,
                             void *stream);
int pvk_resynth_scan_curve(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks, const int32_t *tstart,
                           const int32_t *tlen, const int64_t *toff, const double *pf, const double *prealph,
                           double sr, int hop, int nfft, int hop_an, double fscale, const double *fcurve,
                           int64_t fcurve_len, void *workspace, int64_t workspace_bytes, double *phase_ws,
                           int64_t phase_ws_len, int64_t h_lo, int64_t h_hi, int64_t *rec, int64_t rec_len,
                           void *stream);
int pvk_nyquist_flags_curve(const double *f, const int32_t *gid, int64_t n, double sr, double fscale,
                            const double *fcurve, int64_t fcurve_len, int npks, uint8_t *flags, int64_t nflags,
                            void *stream);

/* ------------------------------------------------------------------ formant gains
 * The magnitudes of a formant-preserving / formant-shifting resynthesis (DESIGN.md 4.3), to be passed as
 * pmag to pvk_resynth_ex / pvk_resynth_render (and their _curve variants).  The envelope of frame row j is
 * the piecewise-linear interpolation L_j of ln(pmag) over the frequencies of the row's points (slots with
 * 0 <= tid < ntracks; knots sorted by frequency, ties by column; held constant beyond the first / last
 * knot, as np.interp).  Every point (f, m) of row j is written as pmag_out[toff[v] + j - tstart[v]] =
 * m * exp(L_j(f * q_j) - L_j(f)), and = m bit for bit where f * q_j == f.  q_j = fscale_j / formant_j, the
 * render's frequency ratio of the row over its formant factor.
 *   tid, ntracks, ntracks_dev, tstart, toff, pf, pmag   as pvk_resynth_ex takes them (ntracks_dev != NULL:
 *                the partial count is read on the device, at most ntracks)
 *   q            the ratio of every row when qcurve = NULL (finite, > 0)
 *   qcurve       device, one ratio per frame row (qcurve_len >= nframes; values the caller's to check)
 *   pmag_out     one double per packed point; a length below min(ntracks, nframes * npks) is rejected,
 *                points at or beyond pmag_out_len are not written
 * Checks its arguments before any CUDA call; allocates nothing.
 */
int pvk_formant_gains(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks, const int32_t *ntracks_dev,
                      const int32_t *tstart, const int64_t *toff, const double *pf, const double *pmag, double q,
                      const double *qcurve, int64_t qcurve_len, double *pmag_out, int64_t pmag_out_len,
                      void *stream);

/* ------------------------------------------------------------------ time map
 * A time-varying time stretch (DESIGN.md 4.3, "Time map"): resample the partials of a packed table onto
 * nrows_out output rows, row b read at the fractional frame tmap[b] = i + u (i = floor(tmap[b])).  For every
 * slot c of row i holding partial v (0 <= tid[i, c] < ntracks), with k = i - tstart[v]:
 *   tid_out[b, c]    = v (ids are kept; -1 for a slot without a point)
 *   f_out, mag_out   = x0 + u * (x1 - x0), x0 / x1 the packed knots k / k + 1 of v (x1 = x0 past its last
 *                      knot), every operation rounded separately (no FMA): u == 0 gives x0 exactly
 *   realph_out       = prealph of knot k
 * Slots without a point get zeros.  The outputs are [nrows_out, npks] frame tables, to be counted with
 * pvk_track_stats and packed with pvk_track_pack (ph = realph_out) for the integrated-phase render.  With a
 * non-decreasing map every partial's output rows form one run, so they are a valid track table; a
 * partial whose rows the map skips is left without points (tlen = 0 after the pack).
 *   tid, ntracks, tstart, tlen, toff, pf, pmag, prealph   the pack of the source table [nframes, npks]
 *   tmap         device, nrows_out float64 frames; the caller checks them (finite, in [0, nframes - 1],
 *                non-decreasing) -- a value outside [0, nframes - 1] gives a row without points
 * Checks sizes, npks and NULL pointers before any CUDA call; allocates nothing.
 */
int pvk_time_map(const int32_t *tid, int64_t nframes, int npks, int64_t ntracks, const int32_t *tstart,
                 const int32_t *tlen, const int64_t *toff, const double *pf, const double *pmag,
                 const double *prealph, const double *tmap, int64_t nrows_out, int32_t *tid_out,
                 double *f_out, double *mag_out, double *realph_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PVK_H_ */
