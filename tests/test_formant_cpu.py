"""CPU: formant gains of the resynthesis (``synth(formant_shift=...)``, ``pvk_formant_gains``) with the
kernels run in the SIMT emulator (tests/emu), against the float64 model of tests/formant_oracle.py:
synthetic tables of 1 to 1024 peaks per row (rows without points, with one, with equal frequencies,
out of order), goldens, sharded windows and clip batches, the host's argument checks, and the effect
on a resynthesised signal's spectrum."""
import os
import sys
import types

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

import formant_oracle as fo
import render_contract as rc
import resynth_emu as rem
from golden_util import case_golden, case_signal
from oracle import pv_oracle as orc
from pypevoc_b200 import pv as P

eh = rem.eh

SEMITONES7 = 2 ** (7 / 12.)


@pytest.fixture(scope="module", autouse=True)
def _build():
    eh.build()


def emu_gains(tid, pk, q, length=None):
    """pvk_formant_gains through the emulator: ``q`` a scalar or one ratio per row."""
    L = eh.lib()
    F, K = tid.shape
    nt = len(pk["tstart"])
    out = np.full(max(len(pk["pmag"]), 1) if length is None else length, np.nan)
    ts = np.ascontiguousarray(pk["tstart"], dtype=np.int32)
    if np.ndim(q) == 0:
        qa = (float(q), None, 0)
    else:
        qc = np.ascontiguousarray(q, dtype=np.float64)
        qa = (1.0, eh.ptr(qc), qc.size)
    eh.check(L.pvk_formant_gains(eh.ptr(np.ascontiguousarray(tid, dtype=np.int32)), F, K, nt, None, eh.ptr(ts),
                                 eh.ptr(pk["toff"]), eh.ptr(pk["pf"]), eh.ptr(pk["pmag"]), *qa, eh.ptr(out), out.size,
                                 None))
    return out[:len(pk["pmag"])]


def check_close(got, ref, rtol=1e-12):
    assert got.shape == ref.shape
    assert np.all(np.isfinite(got))
    err = np.max(np.abs(got - ref) / np.abs(ref)) if ref.size else 0.0
    assert err <= rtol, err
    return err


def point_table(F, K, seed):
    """A ``make_table`` peak table with every peak its own partial (the gains do not look at the
    partials' lengths), and rows of every kind the kernel must handle: no point, one point, equal
    frequencies, columns out of frequency order, a gap in the middle of a row."""
    t = rc.make_table(F, K, rc.SR, seed=seed, stationary=K > 64)
    f, mag = t["f"], t["mag"]
    f[:, 0] = np.where(mag[:, 0] > 0, f[:, 0], 0.0)
    mag[0, :] = 0.0
    if K > 1:
        mag[1, 1:] = 0.0                                          # one knot
        mag[1, 0], f[1, 0] = 0.5, 300.0
    if F > 2:
        mag[2] = np.where(mag[2] > 0, mag[2], 0.01)
        f[2] = np.where(f[2] > 0, f[2], 1000.0)
        if K > 2:
            f[2, K // 2:] = f[2, :K - K // 2]                         # duplicate frequencies
    rng = np.random.default_rng(seed)
    if F > 3:
        mag[3] = np.where(mag[3] > 0, mag[3], 0.02)
        f[3] = np.where(f[3] > 0, f[3], 2000.0)
        perm = rng.permutation(K)
        f[3], mag[3] = f[3, perm], mag[3, perm]                   # shuffled row
    if F > 4 and K > 2:
        mag[4, K // 3] = 0.0                                      # a gap inside the row
    tid = np.where(mag > 0, np.arange(F * K).reshape(F, K), -1).astype(np.int32)
    return rem.pack(tid, f, mag, t["realph"]) + (f, mag, t["realph"])


@pytest.mark.parametrize("K", [1, 3, 50, 400, 1024])
def test_kernel_matches_oracle_synthetic(K):
    F = 8 if K >= 400 else 24
    tid, pk, f, mag, _ = point_table(F, K, seed=K)
    assert (tid[0] < 0).all() and (tid[1] >= 0).sum() == (1 if K > 1 else tid[1, 0] >= 0)
    curve = 0.6 + 0.9 * np.random.default_rng(K).random(F)
    for q in (1.5, 1 / 1.3, curve):
        check_close(emu_gains(tid, pk, q), fo.gained_packed(tid, pk, q))


@pytest.mark.parametrize("name", ["metric_1s", "real_speech", "cfg5_like"])
def test_kernel_matches_oracle_goldens(name):
    g = case_golden(name)
    tr = eh.track(g["f"], g["mag"])
    tid, pk = rem.pack(np.ascontiguousarray(tr["tid"][0]), g["f"], g["mag"], g["realph"])
    F = tid.shape[0]
    sr = float(g["sr"]) if "sr" in g.files else case_signal(name)[1]
    vib = rc.vibrato(F, int(g["hop"]), sr)
    for q in (1.5, 1.0 / SEMITONES7, vib / 1.2):
        check_close(emu_gains(tid, pk, q), fo.gained_packed(tid, pk, q))


def test_equal_ratio_keeps_magnitudes_bit_for_bit():
    """formant_shift = fscale (scalar or curve) and formant_shift = 1 with phase_preserve give q = 1
    exactly, which keeps every magnitude; a curve with r_j == formant_j on some rows keeps those rows."""
    tid, pk, f, mag, _ = point_table(20, 12, seed=5)
    F = tid.shape[0]
    r = rc.vibrato(F, 256, rc.SR, semis=3.0)
    assert P.formant_ratio(False, 1.5, 1.5) == 1.0
    assert P.formant_ratio(True, 1.0, 1.0) == 1.0
    assert np.all(P.formant_ratio(False, r, r) == 1.0)
    assert np.array_equal(emu_gains(tid, pk, 1.0), pk["pmag"])
    assert np.array_equal(emu_gains(tid, pk, P.formant_ratio(False, r, r)), pk["pmag"])
    phi = np.where(np.arange(F) % 2 == 0, r, 1.0)
    q = P.formant_ratio(False, r, phi)
    got = emu_gains(tid, pk, q)
    even = np.zeros(len(pk["pmag"]), dtype=bool)                 # the packed points of the even rows
    for j in range(0, F, 2):
        v = tid[j, tid[j] >= 0].astype(np.int64)
        even[pk["toff"][v] + j - pk["tstart"][v]] = True
    assert np.array_equal(got[even], pk["pmag"][even])
    assert not np.array_equal(got[~even], pk["pmag"][~even])
    check_close(got, fo.gained_packed(tid, pk, q))


@pytest.mark.parametrize("world", [2, 3, 5])
@pytest.mark.parametrize("mode", ["preserve", "free"])
@pytest.mark.parametrize("curve", [False, True])
def test_sharded_equals_unsharded(world, mode, curve):
    """Each rank computes the gains of its window rows from its window tables alone: they equal the
    unsharded gains bit for bit at every point, and the concatenated own signals equal the unsharded
    render bit for bit (simulated ranks of tests/resynth_emu.py)."""
    g, sr, nfft, hop_an, tid, pk = rem.golden_tracked("cfg3_clip")
    F, K = tid.shape
    fscale = 1.0 if mode == "preserve" else SEMITONES7
    phi = 1.0 / (1.0 + 0.2 * np.sin(np.arange(F) / 7.0)) if curve else 1.25
    q = P.formant_ratio(mode == "preserve", fscale, phi, F)
    gains = emu_gains(tid, pk, q)
    gmag = fo.gained_table(tid, g["f"], g["mag"], 1.0)                # [F, K] with every point's gain below
    rows, cols = np.nonzero(tid >= 0)
    v = tid[rows, cols].astype(np.int64)
    gmag[rows, cols] = gains[pk["toff"][v] + rows - pk["tstart"][v]]
    plans = rem.plans_for(F, nfft, hop_an, world, 1.0, 3)
    for p in plans:
        w0, w1 = p["w0"], p["w1"]
        if w1 <= w0:
            continue
        tl, pl = rem.pack(tid[w0:w1], g["f"][w0:w1], g["mag"][w0:w1], g["realph"][w0:w1])
        ql = q[w0:w1] if np.ndim(q) else q
        gl = emu_gains(tl, pl, ql)
        r_, c_ = np.nonzero(tl >= 0)
        vl = tl[r_, c_].astype(np.int64)
        assert np.array_equal(gl[pl["toff"][vl] + r_ - pl["tstart"][vl]], gmag[w0:w1][r_, c_])
    hop = 2 * hop_an
    pp = mode == "preserve"
    ref = rem.render(tid, pk, sr, hop, nfft, hop_an, 1.0, 3, pp, fscale, pmag=gains)
    sig, _ = rem.sharded(tid, g["f"], gmag, g["realph"], sr, hop, nfft, hop_an, 1.0, 3, fscale, world, plans=plans,
                         phase_preserve=pp)
    assert not np.array_equal(gains, pk["pmag"])
    assert sig.shape == ref.shape
    assert np.array_equal(sig, ref), np.max(np.abs(sig - ref))


def test_batch_equals_clips_one_at_a_time():
    """Clips stacked with zero guard rows and the batch's ratio rows (guard rows at 1): the gains of the
    flattened table are those of each clip alone, bit for bit."""
    F, K, G = 16, 10, 3
    clips = [point_table(F, K, seed=s) for s in (11, 12, 13)]
    r = np.stack([rc.vibrato(F, 256, rc.SR, rate=3.0 + s) for s in range(3)])
    phi = np.stack([np.linspace(0.8, 1.3, F) * (1 + 0.1 * s) for s in range(3)])
    q = r / phi
    ff = np.zeros((3, F + G, K))
    mm = np.zeros((3, F + G, K))
    for c, (tid, pk, f, mag, _) in enumerate(clips):
        ff[c, :F], mm[c, :F] = f, mag
    flat_tid = np.where(mm > 0, np.arange(mm.size).reshape(mm.shape), -1).reshape(-1, K).astype(np.int32)
    tidb, pkb = rem.pack(flat_tid, ff.reshape(-1, K), mm.reshape(-1, K), np.zeros((3 * (F + G), K)))
    rows = np.ones((3, F + G))
    rows[:, :F] = q
    gb = emu_gains(tidb, pkb, rows.reshape(-1))
    for c, (tid, pk, f, mag, _) in enumerate(clips):
        g1 = emu_gains(tid, pk, q[c])
        rr, cc = np.nonzero(tid >= 0)
        vb = tidb[c * (F + G) + rr, cc].astype(np.int64)
        v1 = tid[rr, cc].astype(np.int64)
        assert np.array_equal(gb[pkb["toff"][vb] + c * (F + G) + rr - pkb["tstart"][vb]],
                              g1[pk["toff"][v1] + rr - pk["tstart"][v1]])


def test_argument_errors():
    with pytest.raises(ValueError):
        P.formant_ratio(False, 1.5, -1.0)
    with pytest.raises(ValueError):
        P.formant_ratio(False, 1.5, 0.0)
    with pytest.raises(ValueError):
        P.formant_ratio(False, 1.5, float("nan"))
    with pytest.raises(ValueError):
        P.formant_ratio(False, 1.5, np.ones(5), nframes=6)                  # length
    with pytest.raises(ValueError):
        P.formant_ratio(False, 1.5, np.ones((2, 3)), nframes=6)             # shape
    with pytest.raises(ValueError):
        P.formant_ratio(True, 1.0, np.array([1.0, np.inf]), nframes=2)
    with pytest.raises(TypeError):
        P.formant_ratio(True, 1.0, True)
    with pytest.raises(TypeError):
        P.formant_ratio(True, 1.0, "1.0")
    assert P.formant_ratio(True, 1.0, None) is None
    assert np.array_equal(P.formant_ratio(False, np.array([1.5, 3.0]), 1.5), [1.0, 2.0])
    # a batch curve must be [nclips, nframes]
    b = P.SinSumBatch.__new__(P.SinSumBatch)
    b._pb = types.SimpleNamespace(nclips=2, nframes=5, rows_per_clip=8, _dev="cpu")
    with pytest.raises(ValueError):
        b._batch_formant(True, 1.0, np.ones(5))
    with pytest.raises(ValueError):
        b._batch_formant(True, 1.0, np.ones((5, 2)))
    assert b._batch_formant(False, 2.0, 4.0) == 0.5
    # the export checks its arguments before any CUDA call
    L = eh.lib()
    tid, pk, f, mag, _ = point_table(6, 4, seed=1)
    n = len(pk["pmag"])
    out = np.zeros(n)
    ts = np.ascontiguousarray(pk["tstart"], dtype=np.int32)
    nt = len(ts)
    qc = np.ones(5)

    def call(npks=4, q=1.5, qcurve=None, qlen=0, olen=n, nframes=6):
        return L.pvk_formant_gains(eh.ptr(tid), nframes, npks, nt, None, eh.ptr(ts), eh.ptr(pk["toff"]), eh.ptr(pk["pf"]),
                                   eh.ptr(pk["pmag"]), q, qcurve, qlen, eh.ptr(out), olen, None)
    assert call() == 0
    for kw in (dict(q=0.0), dict(q=-1.0), dict(q=float("nan")), dict(q=float("inf")), dict(npks=0), dict(npks=1025),
               dict(qcurve=eh.ptr(qc), qlen=5), dict(olen=min(nt, 24) - 1), dict(nframes=-1)):
        assert call(**kw) != 0, kw
        assert b"pvk_formant_gains" in L.pvk_last_error()


# ------------------------------------------------------------------ behaviour
SR_B, F0_B, NFFT_B, HOP_B = 16000.0, 110.0, 2048, 512
RES = ((500.0, 1.0), (1500.0, 0.5), (2500.0, 0.25))


def envelope(f):
    """Resonance envelope of the test signal: three resonances (500 / 1500 / 2500 Hz) over a floor."""
    f = np.asarray(f, dtype=np.float64)
    return 0.02 + sum(a / (1.0 + ((f - fc) / 120.0) ** 2) for fc, a in RES)


def _envelope_misfit(x):
    """Worst |ln| ratio of the harmonic peaks of the middle frames of ``x`` to ``envelope`` (after the
    best common scale factor), over peaks from 50 Hz to 2.7 kHz: the test signal's top harmonic, above
    which the envelope of a row is held at its last knot."""
    a = orc.analyze(x, SR_B, nfft=NFFT_B, hop=HOP_B, npks=60)
    f, m = a["f"], a["mag"]
    F = f.shape[0]
    sel = slice(F // 4, 3 * F // 4)
    ff, mm = f[sel].ravel(), m[sel].ravel()
    keep = (mm > 0) & (ff > 50.0) & (ff < 2700.0)
    d = np.log(mm[keep]) - np.log(envelope(ff[keep]))
    d -= np.median(d)
    return float(np.max(np.abs(d)))


# measured on the emulated kernels: 0.19 with formant_shift=1.0, 1.74 without (fscale 1.5)
FORMANT_MARGIN = 0.4


def test_formant_preservation_follows_the_envelope():
    """A harmonic signal whose amplitudes follow ``envelope`` is analysed, shifted up by 1.5 with
    integrated phase and analysed again.  With formant_shift = 1 the shifted harmonics keep following
    ``envelope`` at their new frequencies; without it they follow envelope(x / 1.5) and miss it by far."""
    t = np.arange(int(SR_B)) / SR_B
    ks = np.arange(1, int(2700.0 // F0_B) + 1)
    rng = np.random.default_rng(3)
    x = sum(envelope(k * F0_B) * np.cos(2 * np.pi * k * F0_B * t + rng.uniform(0, 2 * np.pi)) for k in ks)
    assert _envelope_misfit(x) < FORMANT_MARGIN / 2                 # the analysis sees the envelope
    a = orc.analyze(x, SR_B, nfft=NFFT_B, hop=HOP_B, npks=40)
    tr = eh.track(a["f"], a["mag"])
    tid, pk = rem.pack(np.ascontiguousarray(tr["tid"][0]), a["f"], a["mag"], a["realph"])
    gains = emu_gains(tid, pk, P.formant_ratio(False, 1.5, 1.0))
    kept = _envelope_misfit(rem.render(tid, pk, SR_B, HOP_B, NFFT_B, HOP_B, fscale=1.5, pmag=gains))
    plain = _envelope_misfit(rem.render(tid, pk, SR_B, HOP_B, NFFT_B, HOP_B, fscale=1.5))
    print("envelope misfit: formant_shift=1.0 %.3f, none %.3f" % (kept, plain))
    assert kept < FORMANT_MARGIN
    assert plain > 3 * FORMANT_MARGIN
