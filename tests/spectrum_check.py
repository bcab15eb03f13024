"""The analysis spectrum (spec_out) against a float64 FFT of the same windowed frames: test signals
and per-frame bounds shared by the emulator and the GPU tests.

The reference of frame j is ``np.fft.fft(x[j hop : j hop + nfft] * win)[:nfft/2]`` in float64,
with ``win`` the fp32 window the kernel reads (win / wfact), so only the FFT's own rounding is
measured.  Per frame, in units of EPS = 2^-24 (fp32 unit roundoff):
  - normwise  ||fx - X||_2 / ||X||_2     <= 6 EPS;
  - per bin   max |fx - X| / max |X|     <= 8 EPS;
  - a frame whose reference is all zero comes out exactly zero.
A radix-2^k FFT of 2^m points in fp32 has a normwise error of a small multiple of EPS that grows
like log2(nfft); measured worst cases are 1.0-2.6 EPS (emulator) from nfft 64 to 8192, so an
error of a few ulps in one twiddle, or a wrong sign on a few of them, is far above the bound."""
import numpy as np

EPS = 2.0 ** -24
NORM_BOUND = 6.0
BIN_BOUND = 8.0
NAMES = ("harmonic", "noise", "impulses")


def signal(name, nfft, hop, nframes, sr=44100, seed=0):
    """float32 signal of exactly ``nframes`` analysis frames.  "harmonic": 29 harmonics of 300 Hz
    plus noise at -60 dB; "noise": white, silent from frame nframes - 2 on (its last two frames are
    all zero); "impulses": a unit impulse every 97 samples (flat spectra: every twiddle of every
    pass shapes every bin)."""
    n = (nframes - 1) * hop + nfft + 1
    rng = np.random.RandomState(seed + nfft)
    if name == "harmonic":
        t = np.arange(n) / sr
        x = sum(np.cos(2 * np.pi * 300.0 * h * t + h) / h for h in range(1, 30)) + 1e-3 * rng.randn(n)
    elif name == "noise":
        x = rng.randn(n)
        x[(nframes - 2) * hop:] = 0.0
    else:
        x = np.zeros(n)
        x[::97] = 1.0
    return x.astype(np.float32)


def frame_errors(fx, x, win, nfft, hop):
    """fx: complex [nframes, nfft/2] of signal x.  Returns (normwise, per-bin) errors per frame in
    units of EPS (NaN for frames whose reference is zero) and the mask of those zero frames."""
    fx = np.asarray(fx)
    nframes = fx.shape[0]
    idx = np.arange(nframes)[:, None] * hop + np.arange(nfft)[None, :]
    X = np.fft.fft(x.astype(np.float64)[idx] * np.asarray(win, dtype=np.float64)[None, :], axis=1)[:, :nfft // 2]
    d = fx.astype(np.complex128) - X
    nx = np.linalg.norm(X, axis=1)
    zero = nx == 0.0
    with np.errstate(divide="ignore", invalid="ignore"):
        norm = np.where(zero, np.nan, np.linalg.norm(d, axis=1) / nx) / EPS
        per_bin = np.where(zero, np.nan, np.abs(d).max(axis=1) / np.abs(X).max(axis=1)) / EPS
    return norm, per_bin, zero


def check(fx, x, win, nfft, hop):
    """Assert the bounds of this module on every frame; returns the worst (normwise, per-bin)."""
    norm, per_bin, zero = frame_errors(fx, x, win, nfft, hop)
    fx = np.asarray(fx)
    assert not fx[zero].any(), "frames with an all-zero reference are not exactly zero: %s" % np.flatnonzero(
        zero & np.asarray(fx).any(axis=1))[:5]
    live = ~zero
    worst = (float(np.max(norm[live])), float(np.max(per_bin[live])))
    assert worst[0] <= NORM_BOUND, ("normwise error %.2f EPS in frame %d" % (worst[0], np.nanargmax(norm)))
    assert worst[1] <= BIN_BOUND, ("per-bin error %.2f EPS max|X| in frame %d" % (worst[1], np.nanargmax(per_bin)))
    return worst
