"""CPU: the per-sample accuracy contract of the resynthesis render (tests/render_contract.py), with the
CUDA sources compiled for the SIMT emulator (tests/emu).  Every case of CASES is a synthetic peak table
tracked, packed and rendered by the emulated kernels, in the three modes (phase-preserving, integrated
phase at a constant ratio, a vibrato curve), and checked sample by sample against the float64
reference.  The cases together reach every branch of the render's dispatch (test_cases_cover_every_branch).

The emulator's ``__cosf`` is libm's ``cosf``, so the bound here (TAU_EMU) covers the fp32 arithmetic of
the render, not the hardware cosine; tests/test_gpu_render_contract.py runs the same cases on the GPU."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

import render_contract as rc
import resynth_emu as rem
import synth_modes_oracle as smo

eh = pytest.importorskip("emu_harness")

TAU_EMU = 2e-6          # the emulated kernels' worst per-sample ratio on these cases is 1.2e-6 (tile16_tpb4)
FLOOR = 1e-9            # absolute: the fp32 accumulator's resolution of the quiet samples


@pytest.fixture(scope="module", autouse=True)
def _build():
    eh.build()


_TABLES = {}


def tracked(name):
    """Synthetic table of a case, tracked and packed by the emulated kernels, and its partials."""
    if name not in _TABLES:
        hop, nfft, hop_an, edge, K, F, minframes, ws_blocks = rc.CASES[name]
        t = rc.make_table(F, K, rc.SR, seed=sum(map(ord, name)), minframes=minframes, stationary=K > 64)
        tr = eh.track(t["f"], t["mag"])
        nt = int(tr["ntracks"][0])
        tid = np.ascontiguousarray(tr["tid"][0])
        pk = eh.track_pack(t["f"], t["mag"], t["ph"], t["realph"], tid, tr["link"][0], nt)
        parts = rc.parts_from_tid(tid, t["f"], t["mag"], t["ph"], t["realph"])
        _TABLES[name] = (t, tid, pk, parts)
    return _TABLES[name]


def run_case(name, label, mode, r):
    hop, nfft, hop_an, edge, K, F, minframes, ws_blocks = rc.CASES[name]
    t, tid, pk, parts = tracked(name)
    w = rem.render(tid, pk, rc.SR, hop, nfft, hop_an, edge, minframes, mode == "preserve", r, ws_blocks=ws_blocks,
                   phase_ws=rem.phase_scratch(pk))
    ref = rc.reference(parts, rc.SR, hop, nfft, hop_an, edge, minframes, mode, r)
    scale = rc.amp_scale(parts, rc.SR, hop, nfft, hop_an, edge, minframes, None if mode == "preserve" else r)
    return rc.check_render(w, ref, scale, TAU_EMU, FLOOR, "%s %s" % (name, label), hop, rc.case_branch(rc.CASES[name]))


@pytest.mark.parametrize("name", sorted(rc.CASES))
def test_emu_render_per_sample(name):
    for label, mode, r in rc.modes(rc.CASES[name], sorted(rc.CASES).index(name)):
        worst = run_case(name, label, mode, r)
        print("%-22s %-11s worst %.2e  %s" % (name, label, worst, rc.branch_label(rc.case_branch(rc.CASES[name]))))


def test_emu_just_under_nyquist():
    """The highest partial at r * max(f) just under sr / 2 is rendered (one ulp more and it is skipped)."""
    name = "g8_G2"
    t, tid, pk, parts = tracked(name)
    fmax = max(np.max(p["f"]) for p in parts)
    fs = np.nextafter(0.5 * rc.SR / fmax, 0.0)
    while fs * fmax >= 0.5 * rc.SR:
        fs = np.nextafter(fs, 0.0)
    assert all(smo.renders(p, rc.SR, 1, False, fs) for p in parts)
    run_case(name, "fscale %.17g" % fs, "free", fs)


def test_generator_tables_are_what_they_say():
    """The tracker finds the partials make_table wrote: starts at row 0, ends at the last row, every
    length from 1 to minframes + 1, frequencies from 1 Hz to 0.49 sr, amplitudes over 1e-4 .. 1e2."""
    t, tid, pk, parts = tracked("tile16_taylor_dE2")
    F = tid.shape[0]
    lens = {len(p["f"]) for p in parts}
    assert {1, 2, 3, 4} <= lens and F in lens
    assert any(p["start_idx"] == 0 for p in parts)
    assert any(p["start_idx"] + len(p["f"]) == F for p in parts)
    fs = np.concatenate([p["f"] for p in parts])
    assert fs.min() < 1.01 and fs.max() == pytest.approx(0.49 * rc.SR)
    ms = np.concatenate([p["mag"] for p in parts])
    assert ms.min() < 1e-3 and ms.max() > 10.0
    # every column's partials are the generator's: one partial per run of filled rows
    runs = sum(int(np.sum(np.diff(np.r_[0, (t["f"][:, c] > 0).astype(int), 0]) == 1)) for c in range(t["f"].shape[1]))
    assert len(parts) == runs
    steep = max(np.max(np.abs(np.diff(p["f"]) / p["f"][:-1])) for p in parts if len(p["f"]) > 1)
    assert steep > 0.02


def test_cases_cover_every_branch():
    """Each branch of the dispatch is reached by at least one case: a new branch, or a case table that
    loses the only case of a branch, fails here."""
    seen = set()
    for name in rc.CASES:
        seen |= rc.branch_features(rc.case_branch(rc.CASES[name]))
    assert rc.BRANCHES <= seen, sorted(rc.BRANCHES - seen)
    assert seen <= rc.BRANCHES, sorted(seen - rc.BRANCHES)


@pytest.mark.parametrize("name", sorted(rc.CASES))
def test_reference_agrees_with_the_models(name):
    """On every case shape the exact-sum reference and the cumsum models of the other tests agree to
    below TAU_EMU / 100 of the local amplitude scale."""
    hop, nfft, hop_an, edge, K, F, minframes, ws_blocks = rc.CASES[name]
    t, tid, pk, parts = tracked(name)
    for label, mode, r in rc.modes(rc.CASES[name], sorted(rc.CASES).index(name)):
        a = rc.reference(parts, rc.SR, hop, nfft, hop_an, edge, minframes, mode, r)
        b = rc.model(parts, rc.SR, hop, nfft, hop_an, edge, minframes, mode, r)
        scale = rc.amp_scale(parts, rc.SR, hop, nfft, hop_an, edge, minframes, None if mode == "preserve" else r)
        rc.check_render(a, b, scale, TAU_EMU / 100, 1e-12, "%s %s" % (name, label), hop)


def extended_body(p, sr, hop, nfft, hop_an, r):
    """Body samples of one partial in integrated-phase mode, the sample-by-sample cumsum of the models
    taken in long double (64-bit significand on x86: 11 more bits than float64)."""
    ld = np.longdouble
    nfr = len(p["f"])
    dfr = nfft / hop_an / 2.
    newt = np.arange(hop * (nfr + dfr))
    fsig = np.interp(newt, hop * (dfr + .5 + np.arange(nfr)), p["f"])[:hop * nfr]
    msig = np.interp(newt, hop * (dfr + np.arange(nfr)), p["mag"])[:hop * nfr]
    rs = np.repeat(np.broadcast_to(np.asarray(r, dtype=np.float64), (nfr,)), hop)
    acc = np.zeros(hop * nfr, dtype=ld)
    acc[1:] = np.cumsum((rs[:-1] * fsig[:-1]).astype(ld))
    th = ld(p["realph"][0]) / (2 * ld(np.pi)) + acc / ld(sr)
    return msig * np.cos(2 * np.pi * (th - np.floor(th)).astype(np.float64))


def test_reference_long_partials():
    """The shape of the long integrated-phase GPU cases (a partial over the 60 s metric prefix: 5168 frames
    at hop 512 and 1024).  There the float64 cumsum of the numpy models drifts by 1e-7 .. 5e-7 of the
    amplitude, so the exact-sum reference is checked against the same cumsum in long double instead:
    they agree to below 1e-8 of the amplitude (the GPU bound / 100).  The block start phases do not
    depend on how the advances are grouped."""
    if np.finfo(np.longdouble).eps > 1e-18:
        pytest.skip("long double is float64 here")
    rng = np.random.default_rng(7)
    sr, nfft, hop_an = 44100.0, 2048, 512
    for nfr, hop in ((5168, 512), (5168, 1024)):
        k = np.arange(nfr)
        pf = 6000.0 + 40.0 * np.sin(2 * np.pi * k / 89.0) + rng.standard_normal(nfr)
        p = dict(start_idx=0, f=pf, mag=np.full(nfr, 0.5), realph=rng.uniform(-np.pi, np.pi, nfr))
        for rr in (1.0, 1.37, rc.vibrato(nfr, hop_an, sr)):
            a = rc.free_synth([p], sr, hop, nfft, hop_an, rr, 1.0, 3)[:hop * nfr]     # the head is cut off
            b = extended_body(p, sr, hop, nfft, hop_an, rr)
            err = np.max(np.abs(a - b)) / 0.5
            print("nfr %d hop %d r %s: reference - long double %.1e" % (nfr, hop, "curve" if np.ndim(rr) else rr, err))
            assert err < 1e-8
    adv = rng.uniform(0.0, 400.0, 5000)
    whole = rc.block_start_phases(0.25, adv)
    tail = rc.block_start_phases(float(whole[2000]), adv[2000:])
    assert np.max(np.abs(whole[2000:] - tail)) < 1e-15


def test_branch_table_restates_the_dispatch():
    """Spot values of render_branch against resynth_run's rules."""
    b = rc.render_branch(512, 50, 2048, 512, 1.0)
    assert (b["kernel"], b["RS"], b["tpb"], b["E"], b["fades"]) == ("tile<16>", 16, 1, 1024, {"taylor"})
    b = rc.render_branch(200, 20, 1024, 256, 1.0)
    assert (b["kernel"], b["nchp"], b["G"], b["windowed"], b["body_slow"]) == ("resynth<8>", 25, 2, False, True)
    b = rc.render_branch(4100, 20, 1024, 256, 0.0)
    assert (b["kernel"], b["nchp"], b["G"], b["windowed"], b["E"]) == ("resynth<16>", 128, 1, True, 0)
    assert rc.render_branch(700, 510, 1024, 256, 1.0)["smem"] is False
    assert rc.render_branch(700, 520, 1024, 256, 1.0)["smem"] is True
    assert rc.render_branch(300, 4, 1024, 256, 1.0, nblocks=40000)["chunks"] == 2
    assert rc.render_branch(512, 4, 1024, 256, 1.0)["fades"] == {"taylor"}       # E 1024
    assert rc.render_branch(512, 4, 1024, 256, 0.1)["fades"] == {"mufu", "partial"}   # E 102
