"""GPU: analyze_warp_kernel (nfft 1024 / 2048: one warp per frame, W frames per CTA sharing a ring of
W + 1 spectrum slots) on the device, through pv.analyze_device.

  - Run structure: run lengths around the group size and a long run, segments that start with a
    warm-up row, clip batches with guard rows (odd clip length, odd hop): every output bit for bit
    equal to the default run sizing, the full signal or the single clip.
  - Selection edges: every bin a candidate, K above the candidate count, exact ties, silence inside
    a signal and a run whose warm-up row is silent.
  - Every emitting case is checked against the oracle run on the kernel's own spectrum.
  - The warp kernel against analyze_kernel (tests/analyze_block_ref.cu, built here with nvcc for
    sm_100a): every output bit for bit.
  - The spectrum against a float64 FFT at every nfft (tests/spectrum_check.py), and two identical
    calls give identical bits."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import pv_oracle as orc
import parity_util as pu
import spectrum_check as sc

pytestmark = pytest.mark.gpu

SR = 44100
W = 8                                  # frames per CTA of analyze_warp_kernel
KEYS = ("f", "mag", "ph", "realph", "binno", "npk", "totalmag")
ALL = KEYS + ("fx", "fine_pos", "fine_val")


@pytest.fixture(scope="module")
def P():
    from pypevoc_b200 import _lib, pv
    _lib.lib()
    return pv


@pytest.fixture(scope="module")
def block_lib(tmp_path_factory):
    import analyze_block_ref as br
    return br.build_gpu(str(tmp_path_factory.mktemp("analyze_block_ref")))


def analyze(P, x, nfft, hop, npks, pkthresh=0.005, **kw):
    """pv.analyze_device on a host or device signal; host copies of every output."""
    xd = x if torch.is_tensor(x) else torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).cuda()
    d = P.analyze_device(xd, SR, nfft, hop, npks, pkthresh, P.host_tables(SR, nfft, hop), **kw)
    return {k: v.cpu().numpy() for k, v in d.items()}


def bits(a):
    a = np.asarray(a)
    if np.iscomplexobj(a):
        a = a.astype(np.complex64)
    return a.view(np.uint8)


def same(a, b, keys, what=""):
    for k in keys:
        assert np.asarray(a[k]).shape == np.asarray(b[k]).shape, (what, k)
        assert np.array_equal(bits(a[k]), bits(b[k])), "%s: %s differs" % (what, k)


def exact(o, nfft, hop, npks, pkthresh, c=0):
    """Kernel logic against the oracle on the kernel's own spectrum (parity_util)."""
    got = {k: o[k][c] for k in KEYS}
    oo = orc.analyze(np.zeros(1), SR, nfft=nfft, hop=hop, npks=npks, pkthresh=pkthresh,
                     fx_given=o["fx"][c].astype(np.complex64))
    pu.compare_exact_on_spectrum(got, oo)
    if "fine_pos" in o:
        fx = o["fx"][c].astype(np.complex64)
        for j in range(fx.shape[0]):
            n = o["npk"][c, j]
            fp, fv = orc.refine_peaks(np.sqrt((fx[j].real * fx[j].real + fx[j].imag * fx[j].imag).astype(np.float64)),
                                      o["binno"][c, j, :n].astype(int))
            assert np.array_equal(fp, o["fine_pos"][c, j, :n]) and np.array_equal(fv, o["fine_val"][c, j, :n]), j
            assert not o["fine_pos"][c, j, n:].any() and not o["fine_val"][c, j, n:].any(), j


def harmonic(nfft, hop, nframes, seed):
    from pypevoc_b200 import signals
    n = (nframes - 1) * hop + nfft + 1
    h = signals.harm(SR, n / SR + 0.01, 170.0 + 35.0 * seed, 60, 0.5, 0.02, seed)[:n]
    return (h + 0.01 * np.random.RandomState(seed).randn(n)).astype(np.float32)


# ---------------------------------------------------------------------------- run structure
@pytest.mark.parametrize("nfft", [1024, 2048])
def test_run_lengths_around_the_group_size(P, nfft):
    """Runs of 1, W - 1, W, W + 1, 2W + 3 and 97 frames give the rows of the default run sizing bit
    for bit, spectrum and refine outputs included."""
    hop, npks = nfft // 4, 40
    x = harmonic(nfft, hop, 150, 1)
    ref = analyze(P, x, nfft, hop, npks, spectra=True, refine=True)
    assert ref["fx"].shape[1] == 150
    exact(ref, nfft, hop, npks, 0.005)
    for run in (1, W - 1, W, W + 1, 2 * W + 3, 97):
        o = analyze(P, x, nfft, hop, npks, run_frames=run, spectra=True, refine=True)
        same(ref, o, ALL, "run %d" % run)


@pytest.mark.parametrize("nfft", [1024, 2048])
def test_segments_without_zero_start_equal_the_full_signal(P, nfft):
    """prev_zero=False: frame0 - 1 is the warm-up row; the segment's rows are the full signal's."""
    hop, npks = nfft // 4 + 1, 30
    x = harmonic(nfft, hop, 5 * W + 3, 2)
    full = analyze(P, x, nfft, hop, npks, spectra=True, refine=True)
    F = full["npk"].shape[1]
    for f0, run in ((1, 0), (5, W + 1), (W, 3), (2 * W + 1, 0), (F - 3, 1)):
        seg = analyze(P, x, nfft, hop, npks, frame0=f0, prev_zero=False, run_frames=run, spectra=True, refine=True)
        same({k: v[:, f0:] for k, v in full.items()}, seg, ALL, "frame0 %d" % f0)


@pytest.mark.parametrize("nfft", [1024, 2048])
def test_clip_batch_with_guard_rows_odd_clip_length(P, nfft):
    """pvk_analyze_batch with an odd clip length (every other clip starts on an odd sample: the
    unaligned frame loads) and an odd hop: every clip's rows, refine outputs included, equal its
    own analysis from an aligned copy; guard rows stay zero."""
    hop, npks, F, G = nfft // 4 + 1, 25, 3 * W + 2, 3
    n = (F - 1) * hop + nfft + 2
    assert n % 2 == 1 and P.n_frames(n, nfft, hop) == F
    x = harmonic(nfft, hop, 4 * W, 3)
    clips = np.stack([x[:n], x[3 * hop + 1:3 * hop + 1 + n], np.zeros(n, np.float32)])
    clips[2, n // 2:] = np.random.RandomState(3).randn(n - n // 2)      # silence, then noise
    xd = torch.from_numpy(clips).cuda()
    assert xd.stride(0) == n
    for run in (0, W - 1):
        b = analyze(P, xd, nfft, hop, npks, out_rows=F + G, run_frames=run, refine=True)
        assert b["fine_pos"].shape == (3, F + G, npks)
        for c in range(3):
            one = analyze(P, xd[c].clone(), nfft, hop, npks, spectra=True, refine=True)
            if run == 0:
                exact(one, nfft, hop, npks, 0.005)
            for k in KEYS + ("fine_pos", "fine_val"):
                assert np.array_equal(bits(b[k][c][:F]), bits(one[k][0])), (run, c, k)
                assert not np.asarray(b[k][c][F:]).any(), (run, c, k)


@pytest.mark.parametrize("nfft", [512, 2048, 4096])
def test_refine_outputs_follow_the_guard_row_layout(P, nfft):
    """refine=True with out_rows > nframes: fine_pos / fine_val are [nclips, out_rows, npks] like the
    other tables, each clip in its own rows (both analysis kernels)."""
    hop, npks, F, G = nfft // 4, 20, 10, 5
    n = (F - 1) * hop + nfft + 1
    rng = np.random.RandomState(nfft)
    clips = np.stack([harmonic(nfft, hop, F, 4)[:n], rng.randn(n).astype(np.float32), harmonic(nfft, hop, F, 5)[:n]])
    xd = torch.from_numpy(clips).cuda()
    b = analyze(P, xd, nfft, hop, npks, out_rows=F + G, refine=True)
    for c in range(3):
        one = analyze(P, xd[c].clone(), nfft, hop, npks, refine=True)
        assert (one["npk"] > 0).all()
        for k in ("fine_pos", "fine_val", "binno", "npk"):
            assert np.array_equal(bits(b[k][c][:F]), bits(one[k][0])), (c, k)
            assert not np.asarray(b[k][c][F:]).any(), (c, k)
    with pytest.raises(AssertionError):
        analyze(P, xd, nfft, hop, npks, out_rows=F + G, spectra=True)
    from pypevoc_b200 import _lib
    L = _lib.lib()
    spec = torch.zeros((3, F + G, nfft // 2), dtype=torch.complex64, device="cuda")
    st = L.pvk_analyze_batch(xd.data_ptr(), 3, n, n, None, None, None, None, nfft, hop, npks, 0.005, 0.0, 0.0, 0, F,
                             1, 0, None, None, None, None, None, None, None, spec.data_ptr(), None, None, F + G, None)
    assert st == 1 and b"spec_out" in L.pvk_last_error()


# ---------------------------------------------------------------------------- selection edges
@pytest.mark.parametrize("nfft", [1024, 2048])
def test_all_bins_candidates_and_large_k(P, nfft):
    """th < 0 (every interior bin a candidate, C = M - 2) with K = C, 100 and 1024; K = 1024 at the
    usual threshold."""
    M = nfft // 2
    hop = nfft // 2 + 1
    x = np.random.RandomState(4).randn(nfft * 12).astype(np.float32)
    for npks, th in ((M - 2, -0.1), (100, -0.1), (1024, -0.1), (1024, 0.005)):
        o = analyze(P, x, nfft, hop, npks, pkthresh=th, spectra=True, refine=True)
        exact(o, nfft, hop, npks, th)


@pytest.mark.parametrize("nfft", [1024, 2048])
def test_exact_ties_path(P, nfft):
    """th < 0 with K between the number of local maxima and C: the boundary bucket is the run of
    equal zero keys of the non-maxima, selected in bin order; all-zero frames tie every bin."""
    M = nfft // 2
    hop = nfft // 2
    x = np.random.RandomState(5).randn(nfft * 8).astype(np.float32)
    x[nfft * 5:] = 0.0
    o = analyze(P, x, nfft, hop, 1, pkthresh=-0.1, spectra=True)
    fx = o["fx"][0].astype(np.complex64)
    pw = fx.real * fx.real + fx.imag * fx.imag
    nmax = ((pw[:, 1:-1] > pw[:, :-2]) & (pw[:, 1:-1] >= pw[:, 2:])).sum(axis=1)
    npks = int(nmax.max()) + 20
    assert npks < M - 2 and int(nmax.min()) == 0
    o = analyze(P, x, nfft, hop, npks, pkthresh=-0.1, spectra=True, refine=True)
    exact(o, nfft, hop, npks, -0.1)


@pytest.mark.parametrize("nfft", [1024, 2048])
def test_silence_inside_a_signal_and_runs_after_silence(P, nfft):
    """Frames 9..12 are all zero: they emit nothing, the frame after them has a zero previous
    spectrum, and a run of 13 frames starts at frame 13 with a silent warm-up row.  Every run length
    gives the default sizing's bits."""
    hop, npks = nfft // 4, 30
    x = harmonic(nfft, hop, 4 * W, 6)
    x[9 * hop:12 * hop + nfft] = 0.0
    ref = analyze(P, x, nfft, hop, npks, spectra=True, refine=True)
    assert not ref["fx"][0][9:13].any() and not ref["npk"][0][9:13].any() and (ref["npk"][0][13:] > 0).all()
    assert not ref["totalmag"][0][9:13].any()
    exact(ref, nfft, hop, npks, 0.005)
    for run in (13, W, 4, 1):
        o = analyze(P, x, nfft, hop, npks, run_frames=run, spectra=True, refine=True)
        same(ref, o, ALL, "run %d" % run)
    seg = analyze(P, x, nfft, hop, npks, frame0=13, prev_zero=False, spectra=True, refine=True)
    same({k: v[:, 13:] for k, v in ref.items()}, seg, ALL, "segment after silence")


# ---------------------------------------------------------------------------- warp kernel = block kernel
def block(L, x, nfft, hop, npks, pkthresh, run_frames):
    """analyze_kernel<LOGM> through pvkt_analyze_block on the device."""
    xd = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).cuda()
    from pypevoc_b200 import pv
    tb = pv.host_tables(SR, nfft, hop)
    dtb = pv._device_tables(tb, xd.device)
    tables = pv._analysis_tables(nfft, xd.device)
    F = pv.n_frames(len(x), nfft, hop)
    out = {k: torch.full((1, F, npks), float("nan"), dtype=torch.float64, device="cuda")
           for k in ("f", "mag", "ph", "realph", "binno", "fine_pos", "fine_val")}
    out["npk"] = torch.full((1, F), -7, dtype=torch.int32, device="cuda")
    out["totalmag"] = torch.full((1, F), float("nan"), dtype=torch.float64, device="cuda")
    spec = torch.zeros((1, F, nfft // 2), dtype=torch.complex64, device="cuda")
    p = lambda t: t.data_ptr()  # noqa: E731
    st = L.pvkt_analyze_block(p(xd), 1, xd.numel(), xd.numel(), p(dtb["win"]), p(dtb["fbin"]), p(dtb["wfbin"]),
                              p(tables), nfft, hop, npks, pkthresh, tb["dt"], tb["fstep"], 0, F, 1, run_frames,
                              p(out["f"]), p(out["mag"]), p(out["ph"]), p(out["realph"]), p(out["binno"]),
                              p(out["npk"]), p(out["totalmag"]), p(spec), p(out["fine_pos"]), p(out["fine_val"]),
                              torch.cuda.current_stream().cuda_stream)
    assert st == 0, L.pvk_last_error()
    out["fx"] = spec
    return {k: v.cpu().numpy() for k, v in out.items()}


@pytest.mark.parametrize("case", ["harmonic", "noise", "all_bins"])
@pytest.mark.parametrize("nfft", [1024, 2048])
def test_warp_kernel_equals_block_kernel(P, block_lib, nfft, case):
    """Every output of the product's analyze_warp_kernel equals analyze_kernel's bit for bit on the
    device, where the FFT's products are fused as compiled: the spectrum, hence binno, npk and
    totalmag, and through the shared peak epilogue f, mag, ph, realph and the refine outputs."""
    M = nfft // 2
    if case == "harmonic":
        hop, npks, th = nfft // 4, 50, 0.005
        x = harmonic(nfft, hop, 6 * W + 5, 7)
    elif case == "noise":
        hop, npks, th = nfft // 4 + 1, 30, 0.005
        x = np.random.RandomState(8).randn(40 * hop + nfft).astype(np.float32)
    else:
        hop, npks, th = M, 100, -0.1
        x = np.random.RandomState(9).randn(30 * M + nfft).astype(np.float32)
    w = analyze(P, x, nfft, hop, npks, pkthresh=th, spectra=True, refine=True)
    b = block(block_lib, x, nfft, hop, npks, th, 5)
    exact(w, nfft, hop, npks, th)
    fw, fb = w["fx"][0].astype(np.complex64), b["fx"][0].astype(np.complex64)
    diff = np.argwhere(fw.view(np.uint64) != fb.view(np.uint64))
    if len(diff):
        j, k = diff[0]
        raise AssertionError("fx differs in %d bins, first at frame %d bin %d: warp %r, block %r"
                             % (len(diff), j, k, fw[j, k], fb[j, k]))
    same(w, b, ALL, "warp vs block")


# ---------------------------------------------------------------------------- spectrum accuracy, determinism
@pytest.mark.parametrize("nfft", [64, 128, 256, 512, 1024, 2048, 4096, 8192])
def test_spectrum_against_float64_fft(P, nfft):
    """spec_out against np.fft.fft in float64 of the same windowed frames, 300 frames per signal,
    odd hop."""
    hop, nframes = nfft // 4 + 1, 300
    win = (P.host_tables(SR, nfft, hop)["win"] / P.host_tables(SR, nfft, hop)["wfact"]).astype(np.float32)
    for name in sc.NAMES:
        x = sc.signal(name, nfft, hop, nframes)
        o = analyze(P, x, nfft, hop, 20, spectra=True)
        assert o["fx"].shape == (1, nframes, nfft // 2)
        worst = sc.check(o["fx"][0], x, win, nfft, hop)
        print("device spectrum nfft %d %s: normwise %.2f, per-bin %.2f (units of 2^-24)" % (nfft, name, *worst))


@pytest.mark.parametrize("nfft", [1024, 2048])
def test_two_identical_calls_give_identical_bits(P, nfft):
    hop, npks = nfft // 4, 50
    x = torch.from_numpy(harmonic(nfft, hop, 400, 9)).cuda()
    a = analyze(P, x, nfft, hop, npks, spectra=True, refine=True)
    b = analyze(P, x, nfft, hop, npks, spectra=True, refine=True)
    same(a, b, ALL, "second call")
