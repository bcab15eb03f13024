"""CPU: the analysis spectrum and the two analysis kernels on the SIMT emulator.

  - At nfft 1024 / 2048 analyze_warp_kernel (one warp per frame) computes every output bit for bit
    as analyze_kernel (one CTA per frame, tests/analyze_block_ref.cu), on every output table.
  - At every nfft the spectrum is within a few fp32 roundings of a float64 FFT of the same frames
    (tests/spectrum_check.py), in every frame and relative to its largest bin.
  - Scaling the signal by 2^s scales fx, mag and totalmag by exactly 2^s and changes no other bit.
  - Clip batches with guard rows: fine_pos / fine_val follow the rows of the other tables.
The emulator computes every product unfused; the device comparisons are in
tests/test_gpu_analyze_warp.py."""
import functools
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

import spectrum_check as sc

eh = pytest.importorskip("emu_harness")
import analyze_block_ref as br  # noqa: E402

SR = 44100
W = 8                                  # frames per CTA of analyze_warp_kernel
KEYS = ("fx", "f", "mag", "ph", "realph", "binno", "npk", "totalmag", "fine_pos", "fine_val")
NFFTS = [64, 128, 256, 512, 1024, 2048, 4096, 8192]


@pytest.fixture(scope="module", autouse=True)
def _build():
    eh.build()
    br.build_emu()


def bits(a):
    """Bit pattern of an output (complex spectra as their fp32 pairs): equality is bit equality,
    -0.0 and NaN included."""
    a = np.asarray(a)
    if np.iscomplexobj(a):
        a = a.astype(np.complex64)
    return a.view(np.uint8)


def assert_bit_equal(a, b, keys=KEYS):
    for k in keys:
        assert np.asarray(a[k]).shape == np.asarray(b[k]).shape, k
        assert np.array_equal(bits(a[k]), bits(b[k])), "%s differs" % k


def _harmonic(nfft, hop, nframes, seed):
    from pypevoc_b200 import signals
    n = (nframes - 1) * hop + nfft + 1
    h = signals.harm(SR, n / SR + 0.01, 190.0 + 30.0 * seed, 40, 0.5, 0.02, seed)[:n]
    return (h + 0.01 * np.random.RandomState(seed).randn(n)).astype(np.float32)


# case -> (signal, hop, npks, pkthresh, warp run length, block run length)
def _case(name, nfft):
    M = nfft // 2
    if name == "harmonic":
        return _harmonic(nfft, nfft // 4, 2 * W + 3, 1), nfft // 4, 40, 0.005, 0, 5
    if name == "noise":
        return np.random.RandomState(7).randn(3 * nfft).astype(np.float32), nfft // 4 + 1, 30, 0.005, 0, 3
    if name == "all_bins_k_below":          # th < 0: every interior bin a candidate, K < C
        return np.random.RandomState(8).randn(5 * nfft).astype(np.float32), M, 100, -0.1, 0, 4
    if name == "all_bins_k_above":          # th < 0, K = 1024 > C = M - 2: no select
        return np.random.RandomState(9).randn(5 * nfft).astype(np.float32), M, 1024, -0.1, 0, 4
    # runs that end on a partial group: 2 W + 3 frames in runs of W + 3 and W (each with its warm-up
    # row: W + 4 and W + 1 local frames, a full group of W and a short last one)
    return _harmonic(nfft, nfft // 4 + 3, 2 * W + 3, 2), nfft // 4 + 3, 25, 0.005, W + 3, 2


@pytest.mark.parametrize("case", ["harmonic", "noise", "all_bins_k_below", "all_bins_k_above", "partial_group"])
@pytest.mark.parametrize("nfft", [1024, 2048])
def test_warp_kernel_equals_block_kernel(nfft, case):
    """Every output of analyze_warp_kernel, the spectrum and fine_pos / fine_val included, equals
    analyze_kernel's bit for bit."""
    x, hop, npks, th, run_w, run_b = _case(case, nfft)
    w = eh.analyze(x, SR, nfft, hop, npks, pkthresh=th, run_frames=run_w, spectra=True, refine=True)
    b = br.analyze_emu(x, SR, nfft, hop, npks, pkthresh=th, run_frames=run_b)
    assert w["nframes"] == b["nframes"] and (w["npk"] > 0).any()
    assert_bit_equal({k: w[k] for k in KEYS}, b)


@functools.lru_cache(maxsize=None)
def _spectrum_run(name, nfft, scale=0):
    hop = nfft // 4 + 1                     # odd hop: unaligned frame starts
    x = sc.signal(name, nfft, hop, 7)
    if scale:
        x = (x * np.float32(2.0 ** scale)).astype(np.float32)
    return x, eh.analyze(x, SR, nfft, hop, 20, spectra=True)


@pytest.mark.parametrize("name", sc.NAMES)
@pytest.mark.parametrize("nfft", NFFTS)
def test_spectrum_against_float64_fft(nfft, name):
    """spec_out against np.fft.fft in float64 of the same windowed frames, frame by frame."""
    hop = nfft // 4 + 1
    x, o = _spectrum_run(name, nfft)
    win = eh.host_tables(SR, nfft, hop)["win_scaled"]
    worst = sc.check(o["fx"][0], x, win, nfft, hop)
    print("nfft %d %s: normwise %.2f, per-bin %.2f (units of 2^-24)" % (nfft, name, worst[0], worst[1]))
    if name == "noise":
        assert not o["fx"][0][-2:].any() and not o["npk"][0][-2:].any()


@pytest.mark.parametrize("s", [-16, 16])
@pytest.mark.parametrize("nfft", NFFTS)
def test_power_of_two_scale_invariance(nfft, s):
    """x 2^s: the same peaks, frequencies and phases bit for bit; fx, mag and totalmag exactly 2^s
    times the unscaled ones.  No threshold hides an absolute constant."""
    for name in ("harmonic", "noise"):
        x, a = _spectrum_run(name, nfft)
        _, b = _spectrum_run(name, nfft, s)
        fx = a["fx"][0].astype(np.complex64)
        comp = np.abs(np.concatenate([fx.real.ravel(), fx.imag.ravel()])).astype(np.float64)
        smallest = comp[comp > 0].min() * 2.0 ** s
        assert smallest ** 2 >= 2.0 ** -126 and comp.max() * 2.0 ** s < 2.0 ** 60   # no subnormal or huge power
        assert (a["npk"] > 0).any()
        for k in ("binno", "npk", "f", "ph", "realph"):
            assert np.array_equal(bits(a[k]), bits(b[k])), (name, k)
        for k in ("fx", "mag", "totalmag"):
            assert np.array_equal(bits(np.asarray(a[k]) * 2.0 ** s), bits(b[k])), (name, k)


@pytest.mark.parametrize("nfft", [512, 2048])
def test_clip_batch_guard_rows_with_refine(nfft):
    """pvk_analyze_batch with refine: fine_pos / fine_val are [nclips, out_rows, npks] like the other
    tables; every clip's rows equal its own analysis and its guard rows stay zero."""
    hop, npks, F, G = nfft // 4, 20, W + 2, 5
    x = _harmonic(nfft, hop, 3 * W, 3)
    n = (F - 1) * hop + nfft + 1
    clips = np.stack([x[:n], x[2 * hop:2 * hop + n], np.random.RandomState(3).randn(n).astype(np.float32)])
    for run in (0, 3):
        b = eh.analyze(clips, SR, nfft, hop, npks, out_rows=F + G, run_frames=run, refine=True)
        assert b["fine_pos"].shape == (3, F + G, npks)
        for c in range(3):
            one = eh.analyze(clips[c], SR, nfft, hop, npks, refine=True)
            assert one["nframes"] == F and (one["npk"] > 0).all()
            for k in ("f", "mag", "ph", "realph", "binno", "npk", "totalmag", "fine_pos", "fine_val"):
                assert np.array_equal(bits(b[k][c][:F]), bits(one[k][0])), (c, k)
                assert not np.asarray(b[k][c][F:]).any(), (c, k)
