"""Numpy model of ``SinSum.synth(phase_preserve=False, fscale=...)``: integrated-phase
resynthesis (pitch shift / time stretch).  The reference's ``RegPartial.synth_no_phase`` fails
before it computes anything (PVAnalysis.py:665), so this model is the specification: it is
``RegPartial.synth`` (:684-756) without the per-block re-anchoring at ``realph`` and with every
frequency scaled by ``fscale``.  The phase is a sample-by-sample ``cumsum`` of the interpolated
frequency over the whole body of a partial, not the kernels' closed form.  With
``phase_preserve=True`` both functions are :mod:`oracle.pv_oracle`'s, unchanged."""
import numpy as np

from oracle import pv_oracle as orc

pi2 = 2.0 * np.pi


def synth_partial(pf, pmag, prealph, sr, hop, overlap, fstep, edge=1.0, phase_preserve=True, fscale=1.0):
    """One partial; returns ``(signal, start_sample)`` like :func:`oracle.pv_oracle.synth_partial`."""
    if phase_preserve:
        if fscale != 1.0:
            raise ValueError("fscale != 1 needs phase_preserve=False")
        return orc.synth_partial(pf, pmag, prealph, sr, hop, overlap, fstep, edge)
    pf = np.asarray(pf, dtype=np.float64)
    pmag = np.asarray(pmag, dtype=np.float64)
    prealph = np.asarray(prealph, dtype=np.float64)
    nfr = len(pf)
    hop = int(hop)
    dfr = 1. / overlap / 2.                                               # :687
    newt = np.arange(hop * (nfr + dfr))                                   # :689
    fsig = np.interp(newt, hop * (dfr + .5 + np.arange(nfr)), pf)         # :701
    msig = np.interp(newt, hop * (dfr + np.arange(nfr)), pmag)            # :702
    n = hop * nfr
    ph = np.empty(n)
    ph[0] = 0.0
    ph[1:] = np.cumsum(fsig[:n - 1])                                      # sum_{m<s} fsig[m]
    ph = prealph[0] + (pi2 * fscale / float(sr)) * ph
    body = msig[:n] * np.cos(ph)
    edgsam = int(dfr * hop * edge)                                        # :740
    q = np.arange(edgsam)
    hmag = msig[0] * (1 - np.cos(np.pi * q / float(edgsam))) / 2.         # :742
    hph = np.flipud(prealph[0] - pi2 * np.cumsum(fscale * pf[0] * np.ones(edgsam) / float(sr)))   # :743-744
    tmag = msig[n] * (1 + np.cos(np.pi * q / float(edgsam))) / 2.         # :748-749
    tph = ph[-1] + pi2 * np.cumsum(fscale * pf[-1] * np.ones(edgsam) / float(sr))                 # :750
    sig = np.concatenate((hmag * np.cos(hph), body, tmag * np.cos(tph)))
    return sig, edgsam


def renders(p, sr, minframes, phase_preserve=True, fscale=1.0):
    """Whether partial ``p`` is rendered: ``minframes`` (:1061) and, with integrated phase, the
    Nyquist rule ``fscale * max(f) < sr / 2``."""
    if len(p["f"]) < minframes:
        return False
    return phase_preserve or fscale * np.max(p["f"]) < 0.5 * sr


def synth(parts, sr, hop, nfft, hop_an, edge=1.0, minframes=3, max_end=None, phase_preserve=True, fscale=1.0):
    """``SinSum.synth`` overlap-add (:1053-1070); output length and placement as in
    :func:`oracle.pv_oracle.synth` (skipped partials still count for ``max_end``)."""
    if phase_preserve:
        if fscale != 1.0:
            raise ValueError("fscale != 1 needs phase_preserve=False")
        return orc.synth(parts, sr, hop, nfft, hop_an, edge, minframes, max_end)
    hop = int(hop)
    dfr = nfft / hop_an / 2.                                              # :1055
    edgsamp = int(edge * hop * dfr)                                       # :1056
    if max_end is None:
        max_end = max(p["start_idx"] + len(p["f"]) - 1 for p in parts)
    w = np.zeros((max_end + 2) * hop + 2 * edgsamp)                       # :1059
    overlap = hop_an / float(nfft)                                        # :824
    fstep = sr / float(nfft)                                              # :825
    for p in parts:
        if renders(p, sr, minframes, False, fscale):
            wi, e = synth_partial(p["f"], p["mag"], p["realph"], sr, hop, overlap, fstep, edge, False, fscale)
            s = int(p["start_idx"] * hop - e) + edgsamp                   # :756,1066
            if s >= 0:
                w[s:s + len(wi)] += wi                                    # :1067-1069
    return w[edgsamp:]                                                    # :1070


def direct_partial(pf, pmag, prealph, sr, hop, overlap, edge=1.0, fscale=1.0):
    """The integrated-phase model evaluated sample by sample with python loops (a check of
    :func:`synth_partial`): returns ``(signal, start_sample)``."""
    pf = [float(v) for v in pf]
    nfr = len(pf)
    hop = int(hop)
    dfr = 1. / overlap / 2.
    E = int(dfr * hop * edge)
    kf = [hop * (dfr + .5 + k) for k in range(nfr)]
    km = [hop * (dfr + k) for k in range(nfr)]
    f = lambda s: float(np.interp(s, kf, pf))                           # noqa: E731
    m = lambda s: float(np.interp(s, km, pmag))                         # noqa: E731
    out = []
    for q in range(E):
        hm = m(0) * (1 - np.cos(np.pi * q / E)) / 2.
        out.append(hm * np.cos(prealph[0] - pi2 * fscale * pf[0] * (E - q) / sr))
    th, acc = float(prealph[0]), 0.0
    for s in range(hop * nfr):
        th = float(prealph[0]) + pi2 * fscale / sr * acc
        out.append(m(s) * np.cos(th))
        acc += f(s)
    for q in range(E):
        tm = m(hop * nfr) * (1 + np.cos(np.pi * q / E)) / 2.
        out.append(tm * np.cos(th + pi2 * fscale * pf[-1] * (q + 1) / sr))
    return np.array(out), E
