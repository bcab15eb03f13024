"""CPU: analyze_warp_kernel (nfft 1024 / 2048: one warp per frame, W frames per CTA sharing a ring of
W + 1 spectrum slots) on the SIMT emulator, over the run structure it has to get right: runs around
a group of W frames, segments that start with a warm-up row, clip batches with guard rows, every bin
a candidate, K above the candidate count and the exact-ties select.  Every case is checked against
the oracle run on the kernel's own spectrum, and the run length, the segment start and the clip
batch must not change a single bit."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

from oracle import pv_oracle as orc
import parity_util as pu

eh = pytest.importorskip("emu_harness")

W = 8                                  # frames per CTA of analyze_warp_kernel (AW in pvk_analyze.cu)
SR = 44100
KEYS = ("f", "mag", "ph", "realph", "binno", "npk", "totalmag")


@pytest.fixture(scope="module", autouse=True)
def _build():
    eh.build()


def _signal(nfft, hop, nframes, seed):
    from pypevoc_b200 import signals
    n = (nframes - 1) * hop + nfft + hop
    h = signals.harm(SR, n / SR + 0.01, 180.0 + 40.0 * seed, 40, 0.5, 0.02, seed)[:n]
    rng = np.random.RandomState(seed)
    return (h + 0.01 * rng.randn(n)).astype(np.float32)


def _exact(o, nfft, hop, npks, pkthresh, c=0):
    got = {k: o[k][c] for k in KEYS}
    oo = orc.analyze(np.zeros(1), SR, nfft=nfft, hop=hop, npks=npks, pkthresh=pkthresh,
                     fx_given=o["fx"][c].astype(np.complex64))
    pu.compare_exact_on_spectrum(got, oo)


def _same(a, b, rows=slice(None), keys=KEYS):
    for k in keys:
        assert np.array_equal(a[k][0][rows], b[k][0]), k


@pytest.mark.parametrize("nfft", [1024, 2048])
def test_run_lengths_around_the_group_size(nfft):
    """Runs of 1, W - 1, W, W + 1 and 2W + 3 frames (short last groups, single-frame runs, runs that
    end exactly on a group) give the rows of the default run sizing, bit for bit, and match the oracle."""
    hop, npks = nfft // 4, 40
    x = _signal(nfft, hop, 3 * W + 5, 1)
    ref = eh.analyze(x, SR, nfft, hop, npks, spectra=True, refine=True)
    _exact(ref, nfft, hop, npks, 0.005)
    for run in (1, W - 1, W, W + 1, 2 * W + 3):
        o = eh.analyze(x, SR, nfft, hop, npks, run_frames=run, spectra=True, refine=True)
        _same(ref, o, keys=KEYS + ("fx", "fine_pos", "fine_val"))


@pytest.mark.parametrize("nfft", [1024, 2048])
def test_segments_without_zero_start_equal_the_full_signal(nfft):
    """prev_zero=0: frame0 - 1 is the warm-up row; the segment's rows are the full signal's rows."""
    hop, npks = nfft // 4, 30
    x = _signal(nfft, hop, 2 * W + 7, 2)
    full = eh.analyze(x, SR, nfft, hop, npks)
    for f0, run in ((1, 0), (5, W + 1), (W + 2, 3)):
        seg = eh.analyze(x, SR, nfft, hop, npks, frame0=f0, prev_zero=0, run_frames=run)
        _same(full, seg, rows=slice(f0, None))


def test_clip_batch_with_guard_rows():
    """pvk_analyze_batch at nfft 2048: every clip's rows equal its own analysis; guard rows stay zero."""
    nfft, hop, npks = 2048, 512, 25
    x = _signal(nfft, hop, 3 * W, 3)
    clips = np.stack([x[:(W + 2) * hop + nfft], x[hop:(W + 3) * hop + nfft], np.zeros((W + 2) * hop + nfft, np.float32)])
    F, G = W + 2, 3
    for run in (0, W - 1):
        b = eh.analyze(clips, SR, nfft, hop, npks, out_rows=F + G, run_frames=run)
        for c in range(3):
            one = eh.analyze(clips[c], SR, nfft, hop, npks)
            for k in KEYS:
                assert np.array_equal(b[k][c][:F], one[k][0]), k
                assert not np.asarray(b[k][c][F:]).any(), k


@pytest.mark.parametrize("nfft", [1024, 2048])
def test_all_bins_candidates_and_large_k(nfft):
    """th < 0: every interior bin is a candidate (C = M - 2), with K below and above C; and K above
    the candidate count at the usual threshold (no select)."""
    M = nfft // 2
    hop = nfft // 2
    x = np.random.RandomState(4).randn(nfft * 5).astype(np.float32)
    for npks, th in ((M - 2, -0.1), (1024, -0.1), (100, -0.1), (1024, 0.005)):
        o = eh.analyze(x, SR, nfft, hop, npks, pkthresh=th, spectra=True, refine=True)
        _exact(o, nfft, hop, npks, th)


@pytest.mark.parametrize("nfft", [1024, 2048])
def test_exact_ties_path(nfft):
    """th < 0 with K between the number of local maxima and C: the boundary bucket is the run of
    exactly equal zero keys of the non-maxima, so only its first entries in bin order are selected.
    An all-zero frame ties every bin."""
    M = nfft // 2
    hop = nfft // 2
    x = np.random.RandomState(5).randn(nfft * 5).astype(np.float32)
    x[nfft * 3:] = 0.0
    o = eh.analyze(x, SR, nfft, hop, 1, pkthresh=-0.1, spectra=True)
    fx = o["fx"][0].astype(np.complex64)
    pw = fx.real * fx.real + fx.imag * fx.imag
    nmax = ((pw[:, 1:-1] > pw[:, :-2]) & (pw[:, 1:-1] >= pw[:, 2:])).sum(axis=1)
    npks = int(nmax.max()) + 20
    assert npks < M - 2 and int(nmax.min()) == 0          # some rows tie on key 0 at the boundary
    o = eh.analyze(x, SR, nfft, hop, npks, pkthresh=-0.1, spectra=True, refine=True)
    _exact(o, nfft, hop, npks, -0.1)


def test_spec_out_and_refine():
    """spec_out holds the untangled spectrum; fine_pos / fine_val are PeakFinder.refine on it."""
    nfft, hop, npks = 1024, 256, 20
    x = _signal(nfft, hop, W + 3, 6)
    a = eh.analyze(x, SR, nfft, hop, npks, spectra=True, refine=True, run_frames=W - 1)
    plain = eh.analyze(x, SR, nfft, hop, npks)
    _same(plain, a)
    fx = a["fx"][0].astype(np.complex64)
    for j in range(a["nframes"]):
        pw = fx[j].real * fx[j].real + fx[j].imag * fx[j].imag
        y = np.sqrt(pw.astype(np.float64))
        n = a["npk"][0, j]
        fp, fv = orc.refine_peaks(y, a["binno"][0, j, :n].astype(int))
        assert np.array_equal(fp, a["fine_pos"][0, j, :n]) and np.array_equal(fv, a["fine_val"][0, j, :n])
        assert not a["fine_pos"][0, j, n:].any() and not a["fine_val"][0, j, n:].any()
    ref = np.fft.fft(x[:nfft].astype(np.float64) * eh.host_tables(SR, nfft, hop)["win_scaled"].astype(np.float64))
    assert np.allclose(a["fx"][0][0], ref[:nfft // 2], rtol=0, atol=1e-5 * np.abs(ref).max())
