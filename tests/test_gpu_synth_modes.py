"""GPU: integrated-phase resynthesis, ``SinSum.synth(phase_preserve=False, fscale=...)``, against
the numpy model (tests/synth_modes_oracle.py), by re-analysis (pitch shift, time stretch), and
path against path (fused / staged / streamed / clip batch) bit for bit."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import parity_util as pu
import synth_modes_oracle as smo
from pypevoc_b200 import signals

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def P():
    from pypevoc_b200 import _lib, pv
    _lib.lib()           # fails loudly if libpvk.so is missing
    return pv


def host_parts(ss):
    h = ss._host_tracks()
    o = h["toff"]
    return [dict(start_idx=int(h["tstart"][v]), f=h["pf"][o[v]:o[v + 1]], mag=h["pmag"][o[v]:o[v + 1]],
                 realph=h["prealph"][o[v]:o[v + 1]]) for v in range(len(h["tstart"]))]


@pytest.fixture(scope="module")
def metric_pv(P):
    """60 s prefix of the benchmark signal (SURVEY 8d recipe), nfft 2048 / hop 512 / npks 50."""
    sr = 44100
    x = signals.harm_torch(sr, 60 * sr, 220.0, 90, 0.5, 0.01, 1, torch.device("cuda"), scale=0.25)
    x = (x * float(np.float32(0.9 / float(x.abs().max())))).cpu().numpy()
    pv = P.PV(x, sr, nfft=2048, hop=512, npks=50, progress=False)
    pv.run_pv()
    return pv


def tone(sr=44100, dur=2.0, f0=220.0, nharm=10):
    t = np.arange(int(sr * dur)) / sr
    return sum(np.sin(2 * np.pi * f0 * h * t + 0.3 * h) / h for h in range(1, nharm + 1)).astype(np.float32) * 0.3


def strongest_freqs(P, x, sr, n=5):
    """Mean frequencies of the ``n`` strongest partials (>= 20 frames) of a fresh analysis, ascending."""
    pv = P.PV(np.asarray(x, dtype=np.float32), sr, nfft=2048, hop=512, npks=20, progress=False)
    pv.run_pv()
    ss = pv.toSinSum()
    h = ss._host_tracks()
    o, tl = h["toff"], h["tlen"]
    keep = [v for v in range(len(tl)) if tl[v] >= 20]
    mags = [h["pmag"][o[v]:o[v + 1]].mean() for v in keep]
    top = [keep[i] for i in np.argsort(mags)[::-1][:n]]
    return np.sort([h["pf"][o[v]:o[v + 1]].mean() for v in top])


def test_metric_prefix_vs_oracle(P, metric_pv):
    ss = metric_pv.toSinSum()
    for hop, fscale in ((512, 1.0), (512, 2 ** (7 / 12.)), (1024, 1.0), (200, 0.8)):
        w = ss.synth(44100, hop, phase_preserve=False, fscale=fscale)
        ref = smo.synth(host_parts(ss), 44100, hop, 2048, 512, phase_preserve=False, fscale=fscale)
        assert w.shape == ref.shape
        snr = pu.snr_db(w, ref)
        print("metric prefix hop %d fscale %.4f: SNR %.1f dB" % (hop, fscale, snr))
        assert snr > 90.0


def test_long_steady_partial_vs_oracle(P):
    """One partial of 120 000 frames: the phase scan runs over ~120 groups and the group-sum scan."""
    nfr, sr, nfft, hop_an = 120000, 44100.0, 2048, 512
    k = np.arange(nfr)
    f = 440.0 + 3.0 * np.sin(2 * np.pi * k / 173.0)
    mag = 0.2 + 0.05 * np.cos(2 * np.pi * k / 911.0)
    realph = np.random.default_rng(5).uniform(-np.pi, np.pi, nfr)
    dev = torch.device("cuda")
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)    # noqa: E731
    pk = dict(tstart=d(np.zeros(1, np.int32)), tlen=d(np.array([nfr], np.int32)), toff=d(np.array([0, nfr], np.int64)),
              pf=d(f), pmag=d(mag), prealph=d(realph))
    tid = d(np.zeros((nfr, 1), np.int32))
    parts = [dict(start_idx=0, f=f, mag=mag, realph=realph)]
    for hop, fscale in ((256, 1.25), (300, 0.9)):
        w = P.resynth_device(tid, pk, sr, hop, nfft, hop_an, phase_preserve=False, fscale=fscale).cpu().numpy()
        ref = smo.synth(parts, sr, hop, nfft, hop_an, phase_preserve=False, fscale=fscale)
        snr = pu.snr_db(w, ref)
        print("long partial hop %d fscale %.2f: SNR %.1f dB" % (hop, fscale, snr))
        assert snr > 90.0


def test_pitch_shift_by_reanalysis(P):
    sr, fs = 44100, 2 ** (5 / 12.)
    x = tone(sr)
    pv = P.PV(x, sr, nfft=2048, hop=512, npks=20, progress=False)
    pv.run_pv()
    y = pv.toSinSum().synth(sr, 512, phase_preserve=False, fscale=fs)
    a, b = strongest_freqs(P, x, sr), strongest_freqs(P, y, sr)
    assert np.all(np.abs(b / (fs * a) - 1) < 1e-3), (a, b)


def test_time_stretch_by_reanalysis(P):
    sr = 44100
    x = tone(sr)
    pv = P.PV(x, sr, nfft=2048, hop=512, npks=20, progress=False)
    pv.run_pv()
    ss = pv.toSinSum()
    y = ss.synth(sr, 1024, phase_preserve=False)
    assert len(y) == P.synth_geometry(max(ss.end), 1024, 2048, 512)[0]
    assert len(y) > 1.9 * len(x)
    a, b = strongest_freqs(P, x, sr), strongest_freqs(P, y, sr)
    assert np.all(np.abs(b / a - 1) < 1e-3), (a, b)


def test_nyquist_rule(P):
    """Harmonics 9 and 10 scaled to >= sr / 2 are left out; the rest equal the model."""
    sr = 44100
    pv = P.PV(tone(sr), sr, nfft=2048, hop=512, npks=20, progress=False)
    pv.run_pv()
    ss = pv.toSinSum()
    fs = 0.5 * sr / (220.0 * 8.5)
    parts = host_parts(ss)
    skipped = [p for p in parts if fs * np.max(p["f"]) >= 0.5 * sr]
    assert len(skipped) >= 2 and len(skipped) < len(parts)
    for hop in (512, 200):
        w = ss.synth(sr, hop, phase_preserve=False, fscale=fs)
        ref = smo.synth(parts, sr, hop, 2048, 512, phase_preserve=False, fscale=fs)
        assert w.shape == ref.shape and pu.snr_db(w, ref) > 90.0


@pytest.mark.parametrize("hop", [512, 200])
def test_paths_bit_identical(P, metric_pv, hop):
    kw = dict(phase_preserve=False, fscale=1.12)
    ss = metric_pv.toSinSum()
    fused = ss.synth(44100, hop, **kw)                   # first call: link + pack + render queued back to back
    staged = ss.synth(44100, hop, **kw)                  # partials known: resynth_device
    assert np.array_equal(fused, staged)
    streamed = ss.synth(44100, hop, hostbuf={}, chunks=8, **kw)
    assert np.array_equal(streamed, fused)
    ss2 = metric_pv.toSinSum()
    streamed_fused = ss2.synth(44100, hop, hostbuf={}, chunks=8, **kw)
    assert np.array_equal(streamed_fused, fused)
    assert np.array_equal(ss.synth(44100, hop, **kw), fused)   # repeatable


def test_clip_batch_equals_single_clips(P):
    import pypevoc_b200 as pb200
    clips = np.stack([signals.speech_like_clip(seed=1000 + i, sr=16000, dur=0.8) for i in range(5)]).astype(np.float32)
    pb = pb200.PVBatch(clips, 16000, nfft=512, hop=128, npks=20)
    pb.run_pv()
    ssb = pb.toSinSum()
    for hop, fs in ((128, 1.3), (200, 0.7)):
        wb = ssb.synth(16000, hop, phase_preserve=False, fscale=fs)
        for i in range(5):
            pv = pb200.PV(clips[i], 16000, nfft=512, hop=128, npks=20, progress=False)
            pv.run_pv()
            w = pv.toSinSum().synth(16000, hop, phase_preserve=False, fscale=fs)
            assert wb[i].shape == w.shape and np.array_equal(wb[i], w), (hop, i)


def test_phase_preserve_unchanged_by_keywords(P, metric_pv):
    ss = metric_pv.toSinSum()
    a = ss.synth(44100, 512)
    assert np.array_equal(a, ss.synth(44100, 512, phase_preserve=True, fscale=1.0))


def test_errors(P, metric_pv):
    ss = metric_pv.toSinSum()
    for bad in (0.0, -1.0, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            ss.synth(44100, 512, phase_preserve=False, fscale=bad)
    with pytest.raises(ValueError):
        ss.synth(44100, 512, phase_preserve=True, fscale=1.5)
    with pytest.raises(TypeError):
        ss.synth(44100, 512, phase_preserve=False, fscale="2")
