"""CPU: integrated-phase resynthesis (``SinSum.synth(phase_preserve=False, fscale=...)``).

The numpy model (tests/synth_modes_oracle.py) against a direct per-sample evaluation, and the
CUDA sources compiled for the SIMT emulator (tests/emu) against the model, through
``pvk_resynth_ex``: every render path (tile kernels for hops that are multiples of 512 / 256 /
128, the staged kernels for other hops), pitch ratios that do and do not trigger the Nyquist
rule, chunked and block-range renders, and argument validation."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

from oracle import pv_oracle as orc
from golden_util import case_golden, case_signal, pv_kwargs
import parity_util as pu
import resynth_emu as rem
import synth_modes_oracle as smo

eh = pytest.importorskip("emu_harness")

GOLDENS = ["two_sines", "readme_vibrato", "cfg3_clip"]


@pytest.fixture(scope="module", autouse=True)
def _build():
    eh.build()


def golden_tracks(name):
    g = case_golden(name)
    _, sr = case_signal(name)
    kw = pv_kwargs(name)
    tr = eh.track(g["f"], g["mag"])
    nt = int(tr["ntracks"][0])
    pk = eh.track_pack(g["f"], g["mag"], g["ph"], g["realph"], tr["tid"][0], tr["link"][0], nt)
    return g, sr, kw, tr["tid"][0], pk, rem.parts(pk)


# ------------------------------------------------------------------ the model
def test_oracle_matches_direct_evaluation():
    rng = np.random.default_rng(3)
    nfr, hop, sr, nfft, hop_an = 6, 48, 8000.0, 256, 64
    pf = 300.0 + 40.0 * rng.standard_normal(nfr)
    pmag = 0.5 + 0.1 * rng.random(nfr)
    prealph = rng.uniform(-np.pi, np.pi, nfr)
    for edge, fscale in ((1.0, 1.0), (0.5, 1.7), (0.0, 0.6)):
        a, ea = smo.synth_partial(pf, pmag, prealph, sr, hop, hop_an / nfft, sr / nfft, edge, False, fscale)
        b, eb = smo.direct_partial(pf, pmag, prealph, sr, hop, hop_an / nfft, edge, fscale)
        assert ea == eb and a.shape == b.shape
        assert np.max(np.abs(a - b)) < 1e-9


def test_oracle_phase_preserve_is_the_existing_model():
    g, sr, kw, tid, pk, parts = golden_tracks("two_sines")
    hop_an = int(g["hop"])
    a = smo.synth(parts, sr, 512, kw["nfft"], hop_an)
    b = orc.synth(parts, sr, 512, kw["nfft"], hop_an)
    assert np.array_equal(a, b)
    with pytest.raises(ValueError):
        smo.synth(parts, sr, 512, kw["nfft"], hop_an, fscale=1.5)


# ------------------------------------------------------------------ emulated kernels vs the model
CASES = []
for _name in GOLDENS:
    for _i, (_hop, _fs) in enumerate([(512, 1.0), (256, 0.5), (128, 1.5), (200, 1.0), (512, 0.5), (256, 1.5),
                                      (128, 1.0), (200, 0.5), (1024, 1.0), (200, 1.5)]):
        CASES.append((_name, _hop, _fs, (0.0, 1.0)[_i % 2], (1, 3)[(_i // 2) % 2]))


@pytest.mark.parametrize("name,hop,fscale,edge,minframes", CASES)
def test_emu_integrated_phase_vs_oracle(name, hop, fscale, edge, minframes):
    g, sr, kw, tid, pk, parts = golden_tracks(name)
    hop_an = int(g["hop"])
    w = rem.render(tid, pk, sr, hop, kw["nfft"], hop_an, edge, minframes, False, fscale)
    ref = smo.synth(parts, sr, hop, kw["nfft"], hop_an, edge, minframes, phase_preserve=False, fscale=fscale)
    assert w.shape == ref.shape
    assert pu.snr_db(w, ref) > 110.0


@pytest.mark.parametrize("name", GOLDENS)
def test_emu_nyquist_rule(name):
    """A ratio that puts some (not all) partials at or above sr / 2: those are absent, the rest match."""
    g, sr, kw, tid, pk, parts = golden_tracks(name)
    hop_an = int(g["hop"])
    fmax = np.array([np.max(p["f"]) for p in parts])
    fs = 0.5 * sr / np.median(fmax)                           # about half of the partials are skipped
    skipped = [fs * m >= 0.5 * sr for m in fmax]
    assert any(skipped) and not all(skipped)
    w = rem.render(tid, pk, sr, 256, kw["nfft"], hop_an, 1.0, 1, False, fs)
    ref = smo.synth(parts, sr, 256, kw["nfft"], hop_an, 1.0, 1, phase_preserve=False, fscale=fs)
    assert pu.snr_db(w, ref) > 110.0
    kept = [p for p, s in zip(parts, skipped) if not s]
    max_end = max(p["start_idx"] + len(p["f"]) - 1 for p in parts)
    ref_kept = smo.synth(kept, sr, 256, kw["nfft"], hop_an, 1.0, 1, max_end=max_end, phase_preserve=False, fscale=fs)
    assert np.array_equal(ref, ref_kept)


def synthetic_long_partial(nfr, hop_an=256, nfft=1024, sr=16000.0, seed=0):
    """One partial of ``nfr`` frames (vibrato + slow amplitude drift), as a one-column track table."""
    rng = np.random.default_rng(seed)
    k = np.arange(nfr)
    f = 700.0 + 25.0 * np.sin(2 * np.pi * k / 97.0) + rng.standard_normal(nfr)
    mag = 0.3 + 0.1 * np.sin(2 * np.pi * k / 531.0)
    realph = rng.uniform(-np.pi, np.pi, nfr)
    tid = np.zeros((nfr, 1), dtype=np.int32)
    pk = dict(tstart=np.zeros(1, dtype=np.int32), tlen=np.array([nfr], dtype=np.int32),
              toff=np.array([0, nfr], dtype=np.int64), pf=f, pmag=mag, prealph=realph)
    return tid, pk, sr, nfft, hop_an


def test_emu_long_partial_spans_scan_groups():
    """~3000 frames: three scan groups of 1024 points, carried through the group-sum scan."""
    tid, pk, sr, nfft, hop_an = synthetic_long_partial(3000)
    parts = rem.parts(pk)
    for hop, fscale in ((256, 1.0), (200, 1.25)):
        w = rem.render(tid, pk, sr, hop, nfft, hop_an, 1.0, 3, False, fscale)
        ref = smo.synth(parts, sr, hop, nfft, hop_an, 1.0, 3, phase_preserve=False, fscale=fscale)
        assert pu.snr_db(w, ref) > 110.0


def test_emu_batch_layout_does_not_change_a_partial():
    """The scanned phases depend on the partial's own points only: a partial placed after others in
    the packed array (shifting its group boundaries) renders to the same bits."""
    tid, pk, sr, nfft, hop_an = synthetic_long_partial(1500, seed=1)
    w1 = rem.render(tid, pk, sr, 256, nfft, hop_an, 1.0, 3, False, 1.1)
    pre = 333                                                 # a short partial in front, in its own column
    F = 1500 + pre
    tid2 = np.full((F, 2), -1, dtype=np.int32)
    tid2[:pre, 1] = 0
    tid2[pre:, 0] = 1
    pk2 = dict(tstart=np.array([0, pre], dtype=np.int32), tlen=np.array([pre, 1500], dtype=np.int32),
               toff=np.array([0, pre, pre + 1500], dtype=np.int64),
               pf=np.concatenate([np.full(pre, 300.0), pk["pf"]]), pmag=np.concatenate([np.zeros(pre), pk["pmag"]]),
               prealph=np.concatenate([np.zeros(pre), pk["prealph"]]))
    w2 = rem.render(tid2, pk2, sr, 256, nfft, hop_an, 1.0, 3, False, 1.1)
    assert np.array_equal(w2[pre * 256:], w1)


@pytest.mark.parametrize("hop", [512, 200])
def test_emu_chunked_and_block_ranges_are_bit_identical(hop):
    g, sr, kw, tid, pk, parts = golden_tracks("cfg3_clip")
    hop_an = int(g["hop"])
    args = (tid, pk, sr, hop, kw["nfft"], hop_an, 1.0, 3, False, 0.75)
    w = rem.render(*args)
    assert np.array_equal(w, rem.render(*args))                              # repeatable
    assert np.array_equal(w, rem.render(*args, ws_blocks=5))                 # small workspace
    assert np.array_equal(w[3 * hop:7 * hop], rem.render(*args, block0=3, nblocks=4))
    # two block ranges, the second reusing the masks, fades and phases of the first
    F, K = tid.shape
    nb = -(-len(w) // hop)
    ws, pws = rem.workspace(F, K, len(pk["tstart"]), nb), rem.phase_scratch(pk)
    a = rem.render(*args, block0=0, nblocks=nb // 2, nout=len(w), ws=ws, phase_ws=pws)
    b = rem.render(*args, block0=nb // 2, nblocks=nb - nb // 2, nout=len(w), ws=ws, phase_ws=pws, reuse_tracks=1)
    assert np.array_equal(w, np.concatenate([a, b]))


def test_emu_phase_preserve_through_ex_is_unchanged():
    g, sr, kw, tid, pk, parts = golden_tracks("two_sines")
    hop_an = int(g["hop"])
    for hop in (512, 200):
        a = eh.resynth(tid, pk, sr, hop, kw["nfft"], hop_an)
        b = rem.render(tid, pk, sr, hop, kw["nfft"], hop_an, phase_preserve=True, phase_ws=np.zeros(0))
        assert np.array_equal(a, b)


@pytest.mark.parametrize("phase_preserve,fscale,pws_len,needle", [
    (0, 0.0, 100, "fscale"), (0, -1.0, 100, "fscale"), (0, float("nan"), 100, "fscale"),
    (0, float("inf"), 100, "fscale"), (1, 1.5, 100, "fscale"), (0, 1.0, None, "phase_ws"),
    (0, 1.0, 1, "phase_ws_len"),
])
def test_ex_rejects_arguments(phase_preserve, fscale, pws_len, needle):
    L = eh.lib()
    F, K, nt = 10, 4, 3
    tid = np.zeros((F, K), dtype=np.int32)
    ts, tl = np.zeros(nt, dtype=np.int32), np.ones(nt, dtype=np.int32)
    toff = np.arange(nt + 1, dtype=np.int64)
    pf = np.full(nt, 100.0)
    out = np.zeros(64)
    ws = np.zeros(1 << 16, dtype=np.uint8)
    pws = None if pws_len is None else np.zeros(pws_len)
    st = L.pvk_resynth_ex(eh.ptr(tid), F, K, nt, None, eh.ptr(ts), eh.ptr(tl), eh.ptr(toff), eh.ptr(pf), eh.ptr(pf),
                          eh.ptr(pf), 16000.0, 16, 64, 16, 1.0, 1, eh.ptr(out), 64, 0, -1, eh.ptr(ws), ws.size, 0,
                          phase_preserve, fscale, eh.ptr(pws), 0 if pws is None else pws.size, None)
    assert st != 0
    msg = L.pvk_last_error().decode()
    assert needle in msg
    assert np.all(out == 0)                                  # nothing was rendered


def test_ex_signature_declared():
    from pypevoc_b200 import _lib
    res, args = _lib.SIGNATURES["pvk_resynth_ex"]
    assert res is C.c_int and len(args) == len(_lib.SIGNATURES["pvk_resynth_dev"][1]) + 4


def test_host_checks_before_the_library():
    from pypevoc_b200.pv import synth_mode
    assert synth_mode() == (True, 1.0)
    assert synth_mode(False, np.float32(1.5)) == (False, 1.5)
    for bad in (0.0, -2.0, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            synth_mode(False, bad)
    with pytest.raises(ValueError):
        synth_mode(True, 1.5)
    for bad in ("2", None, True, 1j):
        with pytest.raises(TypeError):
            synth_mode(False, bad)
