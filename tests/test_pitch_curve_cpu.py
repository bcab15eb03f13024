"""CPU: time-varying pitch shift, ``SinSum.synth(phase_preserve=False, fscale=curve)`` with one ratio per
analysis frame.  The numpy model (tests/synth_curve_oracle.py) against a python-loop evaluation, and
the CUDA sources compiled for the SIMT emulator (tests/emu) against the model through the ``_curve``
exports: every render path, a glide, a vibrato and a step curve, a constant curve equal to the scalar
ratio bit for bit, chunked / block-range renders, a clip batch, the point-wise Nyquist rule, sharded
ranks (simulated one after another) and the argument checks."""
import numpy as np
import pytest
import torch

import resynth_emu as rem
import synth_curve_oracle as sco
import parity_util as pu
from pypevoc_b200 import dist as D
from pypevoc_b200 import pv as P

eh = rem.eh


@pytest.fixture(scope="module", autouse=True)
def _build():
    eh.build()


def curve(kind, F, hop_an, sr):
    """Ratios of the frame rows from their input time t = row * hop_an / sr."""
    t = np.arange(F) * hop_an / sr
    T = max(t[-1], 1e-9)
    if kind == "glide":                                       # one octave down to up
        return 2.0 ** (t / T - 0.5)
    if kind == "vibrato":                                     # +-1 semitone, 5 Hz
        return 2.0 ** (np.sin(2 * np.pi * 5.0 * t) / 12.0)
    if kind == "step":                                        # alternate 0.75 / 1.3 every 7 rows
        return np.where((np.arange(F) // 7) % 2 == 0, 0.75, 1.3)
    raise ValueError(kind)


# ------------------------------------------------------------------ the model
def test_oracle_matches_direct_evaluation():
    rng = np.random.default_rng(5)
    nfr, hop, sr, nfft, hop_an = 7, 40, 8000.0, 256, 64
    pf = 300.0 + 40.0 * rng.standard_normal(nfr)
    pmag = 0.5 + 0.1 * rng.random(nfr)
    prealph = rng.uniform(-np.pi, np.pi, nfr)
    for edge in (1.0, 0.5, 0.0):
        rp = rng.uniform(0.5, 1.8, nfr)
        a, ea = sco.synth_partial(pf, pmag, prealph, sr, hop, hop_an / nfft, rp, edge)
        b, eb = sco.direct_partial(pf, pmag, prealph, sr, hop, hop_an / nfft, rp, edge)
        assert ea == eb and a.shape == b.shape
        assert np.max(np.abs(a - b)) < 1e-9


def test_oracle_constant_curve_is_the_scalar_model():
    g, sr, nfft, hop_an, tid, pk = rem.golden_tracked("cfg3_clip")
    a, b = sco.constant_is_scalar(rem.parts(pk), sr, 256, nfft, hop_an, 1.25, tid.shape[0])
    assert a.shape == b.shape and np.max(np.abs(a - b)) < 1e-8


# ------------------------------------------------------------------ emulated kernels vs the model
CASES = [(name, hop, kind, (i + j) % 2) for name in ("cfg3_clip", "metric_1s")
         for i, hop in enumerate((512, 256, 128, 200)) for j, kind in enumerate(("glide", "vibrato", "step"))]


@pytest.mark.parametrize("name,hop,kind,edge", CASES)
def test_emu_curve_vs_oracle(name, hop, kind, edge):
    g, sr, nfft, hop_an, tid, pk = rem.golden_tracked(name)
    r = curve(kind, tid.shape[0], hop_an, sr)
    w = rem.render(tid, pk, sr, hop, nfft, hop_an, float(edge), fscale=r)
    ref = sco.synth(rem.parts(pk), sr, hop, nfft, hop_an, r, float(edge), 3)
    assert w.shape == ref.shape
    assert pu.snr_db(w, ref) > 110.0


@pytest.mark.parametrize("hop", [512, 256, 128, 200])
def test_emu_constant_curve_is_the_scalar_bit_for_bit(hop):
    g, sr, nfft, hop_an, tid, pk = rem.golden_tracked("cfg3_clip")
    for c in (1.0, 0.8, 1.5):
        a = rem.render(tid, pk, sr, hop, nfft, hop_an, fscale=np.full(tid.shape[0], c))
        b = rem.render(tid, pk, sr, hop, nfft, hop_an, fscale=c)
        assert np.array_equal(a, b), (hop, c)


def test_emu_null_curve_is_the_scalar_export():
    g, sr, nfft, hop_an, tid, pk = rem.golden_tracked("cfg3_clip")
    L = eh.lib()
    F, K = tid.shape
    nt = len(pk["tstart"])
    nout, _ = D.P.synth_geometry(rem.max_end(tid), 256, nfft, hop_an, 1.0)
    out = np.full(nout, np.nan)
    ws = np.zeros(int(L.pvk_resynth_workspace_bytes(F, K, nt, -(-nout // 256))), dtype=np.uint8)
    pws = np.full(len(pk["pf"]), np.nan)
    eh.check(L.pvk_resynth_ex_curve(eh.ptr(tid), F, K, nt, None, eh.ptr(pk["tstart"]), eh.ptr(pk["tlen"]),
                                    eh.ptr(pk["toff"]), eh.ptr(pk["pf"]), eh.ptr(pk["pmag"]), eh.ptr(pk["prealph"]),
                                    float(sr), 256, nfft, hop_an, 1.0, 3, eh.ptr(out), nout, 0, -1, eh.ptr(ws), ws.size,
                                    0, 0, 1.3, None, 0, eh.ptr(pws), pws.size, None))
    assert np.array_equal(out, rem.render(tid, pk, sr, 256, nfft, hop_an, fscale=1.3))


@pytest.mark.parametrize("hop", [512, 200])
def test_emu_chunked_block_ranges_and_reuse_are_bit_identical(hop):
    g, sr, nfft, hop_an, tid, pk = rem.golden_tracked("cfg3_clip")
    r = curve("vibrato", tid.shape[0], hop_an, sr)
    w = rem.render(tid, pk, sr, hop, nfft, hop_an, fscale=r)
    assert np.array_equal(w[3 * hop:7 * hop], rem.render(tid, pk, sr, hop, nfft, hop_an, fscale=r, block0=3, nblocks=4,
                                                         nout=len(w)))
    F, K = tid.shape
    nb = -(-len(w) // hop)
    assert np.array_equal(w, rem.render(tid, pk, sr, hop, nfft, hop_an, fscale=r, ws_blocks=5))
    ws, pws = rem.workspace(F, K, len(pk["tstart"]), nb), rem.phase_scratch(pk)
    a = rem.render(tid, pk, sr, hop, nfft, hop_an, fscale=r, block0=0, nblocks=nb // 2, nout=len(w), ws=ws,
                   phase_ws=pws)
    b = rem.render(tid, pk, sr, hop, nfft, hop_an, fscale=r, block0=nb // 2, nblocks=nb - nb // 2, nout=len(w), ws=ws,
                   phase_ws=pws, reuse_tracks=1)
    assert np.array_equal(w, np.concatenate([a, b]))


def test_emu_batch_equals_clips_alone():
    """Two clips in one flattened table with guard rows (ratio 1 there): each clip's rows of the batch
    render equal the clip rendered alone."""
    g, sr, nfft, hop_an, tid0, _ = rem.golden_tracked("cfg3_clip")
    F, K = tid0.shape
    guard, hop = 8, 256
    R = F + guard
    f = np.zeros((2 * R, K))
    mag, realph = np.zeros_like(f), np.zeros_like(f)
    tid = np.full((2 * R, K), -1, dtype=np.int32)
    nt0 = int(tid0.max()) + 1
    for c, (shift, scale) in enumerate(((0, 1.0), (nt0, 0.9))):
        f[c * R:c * R + F] = g["f"] * scale
        mag[c * R:c * R + F], realph[c * R:c * R + F] = g["mag"], g["realph"]
        tid[c * R:c * R + F] = np.where(tid0 >= 0, tid0 + shift, -1)
    tidb, pkb = rem.pack(tid, f, mag, realph)
    curves = [curve("glide", F, hop_an, sr), curve("step", F, hop_an, sr)]
    rows = np.ones((2, R))
    rows[:, :F] = curves
    wb = rem.render(tidb, pkb, sr, hop, nfft, hop_an, fscale=rows.reshape(-1), nout=2 * R * hop)
    for c in range(2):
        t1, pk1 = rem.pack(tid[c * R:(c + 1) * R], f[c * R:(c + 1) * R], mag[c * R:(c + 1) * R],
                          realph[c * R:(c + 1) * R])
        w1 = rem.render(t1, pk1, sr, hop, nfft, hop_an, fscale=rows[c])
        assert np.array_equal(wb[c * R * hop:c * R * hop + len(w1)], w1), c


def test_emu_nyquist_rule_in_one_frame():
    """Partial 0 crosses sr / 2 in one frame only (the curve's peak there), partial 1 never: partial 0
    is absent, partial 1 renders; without the peak both render."""
    F, K, hop_an, nfft, sr, hop = 40, 2, 256, 1024, 16000.0, 256
    rng = np.random.default_rng(2)
    f = np.stack([np.full(F, 3000.0), np.full(F, 1000.0)], axis=1) + rng.standard_normal((F, 2))
    mag = np.full((F, K), 0.3)
    realph = rng.uniform(-np.pi, np.pi, (F, K))
    tid = np.tile(np.arange(K, dtype=np.int32), (F, 1))
    tid, pk = rem.pack(tid, f, mag, realph)
    r = np.full(F, 1.1)
    r[17] = 2.7                                               # 2.7 * 3000 > 8000; 2.7 * 1000 < 8000
    parts = rem.parts(pk)
    assert [sco.renders(p, sr, 3, r) for p in parts] == [False, True]
    w = rem.render(tid, pk, sr, hop, nfft, hop_an, fscale=r)
    ref = sco.synth(parts, sr, hop, nfft, hop_an, r, 1.0, 3)
    assert pu.snr_db(w, ref) > 110.0
    assert np.array_equal(ref, sco.synth(parts[1:], sr, hop, nfft, hop_an, r, 1.0, 3, max_end=F - 1))
    r2 = r.copy()
    r2[17] = 1.1
    assert all(sco.renders(p, sr, 3, r2) for p in parts)
    w2 = rem.render(tid, pk, sr, hop, nfft, hop_an, fscale=r2)
    assert pu.snr_db(w2, sco.synth(parts, sr, hop, nfft, hop_an, r2)) > 110.0


# ------------------------------------------------------------------ sharded ranks
def boundary_curve(F, plans, hop_an, sr):
    """A vibrato times a step at every rank boundary, so the ratio changes across each of them."""
    r = curve("vibrato", F, hop_an, sr)
    for p in plans[1:]:
        r[p["j0"]:] *= (1.2 if p["rank"] % 2 else 1 / 1.2)
    return r


@pytest.mark.parametrize("name,world", [(n, w) for n in ("cfg3_clip", "metric_1s") for w in (2, 3, 5)])
def test_emu_sharded_curve_equals_unsharded(name, world):
    g, sr, nfft, hop_an, tid, pk = rem.golden_tracked(name)
    F = tid.shape[0]
    r = boundary_curve(F, rem.plans_for(F, nfft, hop_an, world, 1.0, 3), hop_an, sr)
    for hop in ((hop_an, 200) if world == 3 else (2 * hop_an,)):
        ref = rem.render(tid, pk, sr, hop, nfft, hop_an, fscale=r)
        sig, ranks = rem.sharded(tid, g["f"], g["mag"], g["realph"], sr, hop, nfft, hop_an, 1.0, 3, r, world)
        assert sum(q["plan"]["nown"] > 0 for q in ranks) == world
        assert sig.shape == ref.shape and np.array_equal(sig, ref), (hop, np.max(np.abs(sig - ref)))


def test_emu_sharded_needs_the_window_rows():
    g, sr, nfft, hop_an, tid, pk = rem.golden_tracked("cfg3_clip")
    F = tid.shape[0]
    r = boundary_curve(F, rem.plans_for(F, nfft, hop_an, 3, 1.0, 3), hop_an, sr)
    ref = rem.render(tid, pk, sr, hop_an, nfft, hop_an, fscale=r)
    sig, _ = rem.sharded(tid, g["f"], g["mag"], g["realph"], sr, hop_an, nfft, hop_an, 1.0, 3, r, 3, window_rows=False)
    assert not np.array_equal(sig, ref)


# ------------------------------------------------------------------ argument checks
def _tiny():
    F, K, nt = 10, 4, 3
    return dict(F=F, K=K, nt=nt, tid=np.zeros((F, K), dtype=np.int32), ts=np.zeros(nt, dtype=np.int32),
                tl=np.ones(nt, dtype=np.int32), toff=np.arange(nt + 1, dtype=np.int64), pf=np.full(nt, 100.0),
                out=np.zeros(64), ws=np.zeros(1 << 16, dtype=np.uint8), pws=np.zeros(100), rec=np.zeros(8, np.int64),
                flags=np.zeros(4, dtype=np.uint8))


def _call(name, fscale, fc, fc_len, pp=0):
    L, a = eh.lib(), _tiny()
    if name in ("pvk_resynth_ex_curve", "pvk_resynth_render_curve"):
        return getattr(L, name)(eh.ptr(a["tid"]), a["F"], a["K"], a["nt"], None, eh.ptr(a["ts"]), eh.ptr(a["tl"]),
                                eh.ptr(a["toff"]), eh.ptr(a["pf"]), eh.ptr(a["pf"]), eh.ptr(a["pf"]), 16000.0, 16, 64, 16,
                                1.0, 1, eh.ptr(a["out"]), 64, 0, -1, eh.ptr(a["ws"]), a["ws"].size, 0, pp, fscale,
                                eh.ptr(fc), fc_len, eh.ptr(a["pws"]), a["pws"].size, None), a
    if name == "pvk_resynth_scan_curve":
        return L.pvk_resynth_scan_curve(eh.ptr(a["tid"]), a["F"], a["K"], a["nt"], eh.ptr(a["ts"]), eh.ptr(a["tl"]),
                                        eh.ptr(a["toff"]), eh.ptr(a["pf"]), eh.ptr(a["pf"]), 16000.0, 16, 64, 16, fscale,
                                        eh.ptr(fc), fc_len, eh.ptr(a["ws"]), a["ws"].size, eh.ptr(a["pws"]),
                                        a["pws"].size, -1, -1, eh.ptr(a["rec"]), a["rec"].size, None), a
    f = np.full(a["F"] * a["K"], 9000.0)
    gid = np.zeros(a["F"] * a["K"], dtype=np.int32)
    return L.pvk_nyquist_flags_curve(eh.ptr(f), eh.ptr(gid), f.size, 16000.0, fscale, eh.ptr(fc), fc_len, a["K"],
                                     eh.ptr(a["flags"]), 4, None), a


EXPORTS = ["pvk_resynth_ex_curve", "pvk_resynth_render_curve", "pvk_resynth_scan_curve", "pvk_nyquist_flags_curve"]


@pytest.mark.parametrize("name", EXPORTS)
@pytest.mark.parametrize("fscale,fc_len,pp,needle", [(1.0, 9, 0, "fcurve_len"), (1.5, 10, 0, "fscale"),
                                                      (1.0, 10, 1, "phase_preserve")])
def test_curve_exports_reject_arguments(name, fscale, fc_len, pp, needle):
    if pp and name not in EXPORTS[:2]:
        pytest.skip("no phase_preserve argument")
    fc = np.full(10, 1.0)
    st, a = _call(name, fscale, fc, fc_len, pp)
    assert st != 0
    assert needle in eh.lib().pvk_last_error().decode()
    assert np.all(a["out"] == 0) and np.all(a["flags"] == 0) and np.all(a["pws"] == 0)


def test_nyquist_flags_curve_rejects_partial_rows_and_flags_per_row():
    L = eh.lib()
    f = np.array([1000.0, 5000.0, 5000.0, 1000.0])
    gid = np.array([0, 1, 2, 3], dtype=np.int32)
    fl = np.zeros(4, dtype=np.uint8)
    r = np.array([1.0, 2.0])
    assert L.pvk_nyquist_flags_curve(eh.ptr(f), eh.ptr(gid), 3, 16000.0, 1.0, eh.ptr(r), 2, 2, eh.ptr(fl), 4, None) != 0
    eh.check(L.pvk_nyquist_flags_curve(eh.ptr(f), eh.ptr(gid), 4, 16000.0, 1.0, eh.ptr(r), 2, 2, eh.ptr(fl), 4, None))
    assert fl.tolist() == [0, 0, 1, 0]                        # row 1 at ratio 2: 10000 >= 8000, 2000 < 8000


def test_curve_signatures_declared():
    from pypevoc_b200 import _lib
    for name, base in (("pvk_resynth_ex_curve", "pvk_resynth_ex"), ("pvk_resynth_render_curve", "pvk_resynth_render"),
                       ("pvk_resynth_scan_curve", "pvk_resynth_scan")):
        assert len(_lib.SIGNATURES[name][1]) == len(_lib.SIGNATURES[base][1]) + 2
    assert len(_lib.SIGNATURES["pvk_nyquist_flags_curve"][1]) == len(_lib.SIGNATURES["pvk_nyquist_flags"][1]) + 3


def test_synth_mode_curve_checks():
    r = np.linspace(0.5, 2.0, 12)
    pp, c = P.synth_mode(False, r, nframes=12)
    assert pp is False and c.dtype == np.float64 and np.array_equal(c, r)
    assert np.array_equal(P.synth_mode(False, list(r))[1], r)
    assert np.array_equal(P.synth_mode(False, torch.tensor(r, dtype=torch.float32))[1], r.astype(np.float32))
    assert np.array_equal(P.synth_mode(False, np.arange(1, 4))[1], [1.0, 2.0, 3.0])
    for bad in (np.ones(3, dtype=bool), np.ones(3, dtype=complex), torch.ones(3, dtype=torch.bool),
                torch.ones(3, dtype=torch.complex64), ["a", "b"], [None, 1.0], np.array([object()])):
        with pytest.raises(TypeError):
            P.synth_mode(False, bad)
    for bad in (np.ones(11), np.ones((3, 4)), np.array(1.5), np.array([1.0, np.nan] * 6), np.array([1.0, np.inf] * 6),
                np.array([1.0, 0.0] * 6), np.array([1.0, -1.0] * 6)):
        with pytest.raises(ValueError):
            P.synth_mode(False, bad, nframes=12)
    with pytest.raises(ValueError):
        P.synth_mode(True, r, nframes=12)
