"""Numpy model of ``SinSum.synth(phase_preserve=False, fscale=r)`` with a curve ``r``: one frequency
ratio per analysis frame (row of the frame table), ``r[b]`` applying to every partial in output block
``b`` (output samples ``[b*hop, (b+1)*hop)``).  For a partial with start frame ``st`` and ``nfr`` frames:

- body: ``theta(s) = realph[0] + 2 pi / sr * sum_{m<s} r[st + m // hop] * fsig[m]``, a
  sample-by-sample ``cumsum`` with a per-sample ratio;
- head: constant frequency ``r[st] * f[0]``, run backwards from ``realph[0]``;
- tail: continues from ``theta(hop * nfr - 1)`` at ``r[st + nfr - 1] * f[-1]``;
- Nyquist rule: not rendered if any point has ``r[st + ii] * f[ii] >= sr / 2``.

Overlap-add, ``minframes`` and the output length are those of :mod:`synth_modes_oracle` (which a
constant curve reproduces)."""
import numpy as np

import synth_modes_oracle as smo

pi2 = 2.0 * np.pi


def synth_partial(pf, pmag, prealph, sr, hop, overlap, rp, edge=1.0):
    """One partial with the ratios ``rp`` of its own rows (``len(rp) == len(pf)``); returns
    ``(signal, start_sample)``."""
    pf = np.asarray(pf, dtype=np.float64)
    pmag = np.asarray(pmag, dtype=np.float64)
    prealph = np.asarray(prealph, dtype=np.float64)
    rp = np.asarray(rp, dtype=np.float64)
    nfr = len(pf)
    assert len(rp) == nfr
    hop = int(hop)
    dfr = 1. / overlap / 2.
    newt = np.arange(hop * (nfr + dfr))
    fsig = np.interp(newt, hop * (dfr + .5 + np.arange(nfr)), pf)
    msig = np.interp(newt, hop * (dfr + np.arange(nfr)), pmag)
    n = hop * nfr
    rs = np.repeat(rp, hop)                                               # ratio of every body sample
    ph = np.empty(n)
    ph[0] = 0.0
    ph[1:] = np.cumsum(rs[:n - 1] * fsig[:n - 1])
    ph = prealph[0] + (pi2 / float(sr)) * ph
    body = msig[:n] * np.cos(ph)
    edgsam = int(dfr * hop * edge)
    q = np.arange(edgsam)
    hmag = msig[0] * (1 - np.cos(np.pi * q / float(edgsam))) / 2.
    hph = np.flipud(prealph[0] - pi2 * np.cumsum(rp[0] * pf[0] * np.ones(edgsam) / float(sr)))
    tmag = msig[n] * (1 + np.cos(np.pi * q / float(edgsam))) / 2.
    tph = ph[-1] + pi2 * np.cumsum(rp[-1] * pf[-1] * np.ones(edgsam) / float(sr))
    return np.concatenate((hmag * np.cos(hph), body, tmag * np.cos(tph))), edgsam


def part_ratios(p, r):
    st = int(p["start_idx"])
    return np.asarray(r, dtype=np.float64)[st:st + len(p["f"])]


def renders(p, sr, minframes, r):
    """``minframes`` (:1061) and the point-wise Nyquist rule at each point's row ratio."""
    if len(p["f"]) < minframes:
        return False
    return bool(np.all(part_ratios(p, r) * np.asarray(p["f"]) < 0.5 * sr))


def synth(parts, sr, hop, nfft, hop_an, r, edge=1.0, minframes=3, max_end=None):
    """Overlap-add as :func:`synth_modes_oracle.synth`; ``r``: one ratio per frame row."""
    hop = int(hop)
    dfr = nfft / hop_an / 2.
    edgsamp = int(edge * hop * dfr)
    if max_end is None:
        max_end = max(p["start_idx"] + len(p["f"]) - 1 for p in parts)
    w = np.zeros((max_end + 2) * hop + 2 * edgsamp)
    overlap = hop_an / float(nfft)
    for p in parts:
        if renders(p, sr, minframes, r):
            wi, e = synth_partial(p["f"], p["mag"], p["realph"], sr, hop, overlap, part_ratios(p, r), edge)
            s = int(p["start_idx"] * hop - e) + edgsamp
            if s >= 0:
                w[s:s + len(wi)] += wi
    return w[edgsamp:]


def direct_partial(pf, pmag, prealph, sr, hop, overlap, rp, edge=1.0):
    """The curve model evaluated sample by sample with python loops (a check of
    :func:`synth_partial`): returns ``(signal, start_sample)``."""
    pf = [float(v) for v in pf]
    rp = [float(v) for v in rp]
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
        out.append(hm * np.cos(prealph[0] - pi2 * rp[0] * pf[0] * (E - q) / sr))
    th, acc = float(prealph[0]), 0.0
    for s in range(hop * nfr):
        th = float(prealph[0]) + pi2 / sr * acc
        out.append(m(s) * np.cos(th))
        acc += rp[s // hop] * f(s)
    for q in range(E):
        tm = m(hop * nfr) * (1 + np.cos(np.pi * q / E)) / 2.
        out.append(tm * np.cos(th + pi2 * rp[-1] * pf[-1] * (q + 1) / sr))
    return np.array(out), E


def constant_is_scalar(parts, sr, hop, nfft, hop_an, c, nframes, edge=1.0, minframes=3):
    """The curve model at ``r[:] = c`` and the scalar model at ``fscale = c`` (for a test)."""
    return (synth(parts, sr, hop, nfft, hop_an, np.full(nframes, c), edge, minframes),
            smo.synth(parts, sr, hop, nfft, hop_an, edge, minframes, phase_preserve=False, fscale=c))
