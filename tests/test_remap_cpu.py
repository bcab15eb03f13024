"""CPU: the remap of the partials (``SinSum.remap(tau)``, ``pvk_track_relink``) with the kernels run in the SIMT
emulator (tests/emu): the relink export, the stats and the pack against the float64 model of
tests/remap_oracle.py bit for bit (1 to 1024 peaks per row, goldens, maps in any order and every map of the
time-map tests), a non-decreasing remap rendered bit for bit as the time map of the same map, a reversal
applied twice, non-monotone renders against the float64 reference of the render contract
(tests/render_contract.py), and the argument checks of the host and of the export."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

import render_contract as rc
import remap_emu as rme
import remap_oracle as rmo
import resynth_emu as rem
import time_map_emu as tme
import time_map_oracle as tmo
from pypevoc_b200 import pv as P
from test_time_map_cpu import TAU_EMU, FLOOR, fake_sinsum, golden, run_table

eh = rem.eh


@pytest.fixture(scope="module", autouse=True)
def _build():
    eh.build()


def check_remap(tid, pk, tau, label=""):
    """The emulated remap (map, relink, stats, pack) against the model, bit for bit."""
    tid_r, link, pkr, (npts, last, nt) = rme.remap_pack(tid, pk, tau)
    ref_tid, ref_link, ref_pk, _ = rmo.remap(tid, pk, tau)
    assert np.array_equal(link, ref_link), label
    assert np.array_equal(tid_r, ref_tid), label
    assert nt == len(ref_pk["tstart"]) and npts == len(ref_pk["pf"]), label
    assert last == (rem.max_end(ref_tid) if nt else -1), label
    rmo.check_pack(pkr, ref_pk)
    return tid_r, pkr


@pytest.mark.parametrize("K", [1, 31, 32, 33, 100, 513, 1024])
def test_relink_matches_model_synthetic(K):
    F = 14 if K > 100 else 30
    tid, pk, _ = run_table(F, K, seed=K)
    for name, tau in rmo.all_maps(F).items():
        check_remap(tid, pk, tau, "K %d %s" % (K, name))


@pytest.mark.parametrize("name", ["real_speech", "real_guitar"])
def test_relink_matches_model_goldens(name):
    _, _, _, tid, pk = golden(name)
    F = tid.shape[0]
    maps = rmo.all_maps(F)
    maps["speed"] = tmo.speed_map(0.8 + 0.45 * (0.5 + 0.5 * np.sin(np.arange(2 * F) * 0.05)), F)
    for label, tau in maps.items():
        check_remap(tid, pk, tau, "%s %s" % (name, label))


def test_jump_back_keeps_persisting_partials():
    """A loop from the last row back to an earlier one: the partials present at both rows continue (the
    link points at their column), the others end or begin there."""
    tid, pk, _ = run_table(30, 12, seed=4)
    j1, j0 = 24, 15
    tau = np.concatenate([np.arange(0.0, j1 + 1.0), np.arange(j0, 30.0)])
    tid_r, link, _, _ = rme.remap_pack(tid, pk, tau)
    b = j1 + 1                                                      # the first output row after the jump
    both = set(tid[j1][tid[j1] >= 0]) & set(tid[j0][tid[j0] >= 0])
    only = set(tid[j0][tid[j0] >= 0]) - both
    assert both and only
    for c in range(12):
        v = tid[j0, c]
        if v in both:
            assert link[b, c] >= 0 and tid[j1, link[b, c]] == v and tid_r[b, c] == tid_r[b - 1, link[b, c]]
        elif v in only:
            assert link[b, c] <= -2 and tid_r[b, c] > tid_r[:b].max()


# ------------------------------------------------------------------ non-decreasing maps: the time map
def compact(tm, pkm):
    """The time map's table with the partials it skips removed and the ids compacted in order."""
    keep = np.asarray(pkm["tlen"]) > 0
    new = np.cumsum(keep) - 1
    tid = np.where(tm >= 0, new[np.maximum(tm, 0)], -1).astype(np.int32)
    o = pkm["toff"]
    pk = dict(tstart=pkm["tstart"][keep], tlen=pkm["tlen"][keep], toff=np.concatenate([[0], np.cumsum(pkm["tlen"][keep])]),
              pf=pkm["pf"], pmag=pkm["pmag"], prealph=pkm["prealph"])
    assert o[-1] == len(pkm["pf"])
    return tid, pk


@pytest.mark.parametrize("K", [1, 33, 100])
def test_monotone_remap_is_the_compacted_time_map(K):
    tid, pk, _ = run_table(30, K, seed=50 + K)
    for name, tau in tmo.example_maps(30).items():
        tm, pkm, last = tme.time_map_pack(tid, pk, tau)
        tid_r, _, pkr, (_, last_r, _) = rme.remap_pack(tid, pk, tau)
        ct, cpk = compact(tm, pkm)
        assert np.array_equal(tid_r, ct), name
        rmo.check_pack(pkr, cpk)
        assert last_r == last


@pytest.mark.parametrize("hop", [256, 512, 200])
def test_monotone_remap_renders_as_the_time_map(hop):
    """For every non-decreasing map, the remapped partials render the bits of the time-mapped ones, with
    scalar and curve fscale and with formant_shift (values and curves)."""
    F, K, nfft, hop_an = 36, 10, 1024, 256
    tid, pk, _ = run_table(F, K, seed=hop + 7)
    maps = dict(tmo.example_maps(F))
    maps["curve"] = tmo.speed_map(0.8 + 0.45 * (np.arange(60) % 20) / 19.0, F)
    for name, tau in maps.items():
        B = len(tau)
        tm, pkm, last = tme.time_map_pack(tid, pk, tau)
        tr, _, pkr, (_, last_r, _) = rme.remap_pack(tid, pk, tau)
        assert last_r == last
        nout = P.synth_geometry(last, hop, nfft, hop_an)[0]
        vib = rc.vibrato(B, hop_an, rc.SR, semis=2.0)
        for r, phi in ((1.0, None), (1.5, None), (vib, None), (1.5, 1.0), (vib, vib[::-1]), (1.0, 0.8)):
            pm = pmr = None
            if phi is not None:
                q = P.formant_ratio(False, r, phi)
                pm, pmr = gains(tm, pkm, q), gains(tr, pkr, q)
            pws = np.full(max(len(pkm["pf"]), len(pkm["tstart"]), 1), np.nan)      # phase scratch, sized as in gains()
            a = rem.render(tm, pkm, rc.SR, hop, nfft, hop_an, fscale=r, pmag=pm, nout=nout, phase_ws=pws)
            b = rem.render(tr, pkr, rc.SR, hop, nfft, hop_an, fscale=r, pmag=pmr, nout=nout)
            assert np.all(np.isfinite(a)) and np.array_equal(a, b), name


def gains(tid, pk, q):
    """pvk_formant_gains through the emulator: the magnitudes a formant-shifting render takes.  The export wants
    min(ntracks, B * K) doubles, which the skipped partials of a time-mapped pack (tlen 0) can make more than
    its points."""
    L = eh.lib()
    F, K = tid.shape
    out = np.full(max(len(pk["pmag"]), len(pk["tstart"]), 1), np.nan)
    if np.ndim(q) == 0:
        qa = (float(q), None, 0)
    else:
        qc = np.ascontiguousarray(q, dtype=np.float64)
        qa = (1.0, eh.ptr(qc), qc.size)
    eh.check(L.pvk_formant_gains(eh.ptr(np.ascontiguousarray(tid, dtype=np.int32)), F, K, len(pk["tstart"]), None,
                                 eh.ptr(pk["tstart"]), eh.ptr(pk["toff"]), eh.ptr(pk["pf"]), eh.ptr(pk["pmag"]), *qa,
                                 eh.ptr(out), out.size, None))
    return out


def partial_set(pk):
    """The partials of a pack as a set of (start, f values, mag values)."""
    return {(int(p["start_idx"]), tuple(p["f"]), tuple(p["mag"])) for p in rem.parts(pk)}


@pytest.mark.parametrize("K", [1, 33, 100])
def test_reverse_twice_gives_back_the_partials(K):
    F = 30
    tid, pk, _ = run_table(F, K, seed=90 + K)
    rev = np.arange(F - 1, -1, -1.0)
    t1, _, p1, _ = rme.remap_pack(tid, pk, rev)
    assert len(p1["tstart"]) == len(pk["tstart"])
    t2, _, p2, _ = rme.remap_pack(t1, p1, rev)
    assert partial_set(p2) == partial_set(pk)
    assert np.array_equal(t2 >= 0, tid >= 0)


# ------------------------------------------------------------------ non-monotone renders
@pytest.mark.parametrize("hop", [256, 512, 200])
def test_remapped_render_matches_reference(hop):
    """Reverse, loop, ping-pong, scrub and jump-back maps, rendered from the remapped pack and checked sample by
    sample against the float64 integrated-phase reference of its partials."""
    F, K, nfft, hop_an = 40, 10, 1024, 256
    tid, pk, _ = run_table(F, K, seed=200 + hop)
    for name, tau in rmo.remap_maps(F).items():
        tr, _, pkr, (_, last, _) = rme.remap_pack(tid, pk, tau)
        nout = P.synth_geometry(last, hop, nfft, hop_an)[0]
        parts = rem.parts(pkr)
        for r in (1.0, rc.vibrato(len(tau), hop_an, rc.SR, semis=2.0)):
            w = rem.render(tr, pkr, rc.SR, hop, nfft, hop_an, fscale=r, nout=nout)
            ref = rc.reference(parts, rc.SR, hop, nfft, hop_an, 1.0, 3, "free", r)
            scale = rc.amp_scale(parts, rc.SR, hop, nfft, hop_an, 1.0, 3, r)
            rc.check_render(w, ref, scale, TAU_EMU, FLOOR, "%s %s" % (name, "curve" if np.ndim(r) else "scalar"), hop)


def test_remapped_golden_render_matches_reference():
    sr, nfft, hop_an, tid, pk = golden("real_speech")
    F = tid.shape[0]
    tau = np.concatenate([np.arange(0.0, F - 1.0, 0.75), np.arange(F - 1.0, 0.0, -1.5)])    # ping-pong
    tr, _, pkr, (_, last, _) = rme.remap_pack(tid, pk, tau)
    w = rem.render(tr, pkr, sr, hop_an, nfft, hop_an, nout=P.synth_geometry(last, hop_an, nfft, hop_an)[0])
    parts = rem.parts(pkr)
    ref = rc.reference(parts, sr, hop_an, nfft, hop_an, 1.0, 3, "free", 1.0)
    scale = rc.amp_scale(parts, sr, hop_an, nfft, hop_an, 1.0, 3, 1.0)
    rc.check_render(w, ref, scale, TAU_EMU, FLOOR, "real_speech ping-pong", hop_an)


# ------------------------------------------------------------------ argument checks
def test_host_checks():
    F = 12
    assert np.array_equal(P.time_map_values([5.0, 2.0, 7.5, 0.0], F, monotone=False), [5.0, 2.0, 7.5, 0.0])
    assert np.array_equal(P.time_map_values(np.arange(F - 1, -1, -1), F, monotone=False), np.arange(F - 1.0, -1, -1))
    with pytest.raises(ValueError, match="non-decreasing"):
        P.time_map_values([0.0, 2.0, 1.0], F)                      # the default keeps its check
    for bad in ([0.0, np.nan], [0.0, np.inf], [-0.5, 1.0], [3.0, F - 1 + 1e-9], [F - 1 + 1e-9, 0.0],
                np.zeros((2, 3)), [], np.zeros(0)):
        with pytest.raises(ValueError):
            P.time_map_values(bad, F, monotone=False)
        with pytest.raises(ValueError):
            fake_sinsum(F, 4).remap(bad)
    for bad in ("0 1 2", 3.0, None, np.array(["a"]), np.array([True, False]), np.array([1 + 1j])):
        with pytest.raises(TypeError):
            P.time_map_values(bad, F, monotone=False)
        with pytest.raises(TypeError):
            fake_sinsum(F, 4).remap(bad)


def test_remapped_sinsum_refuses_phase_preserve_before_any_launch():
    ss = fake_sinsum(12, 4)
    ss._remapped = True
    for kw in (dict(), dict(phase_preserve=True), dict(phase_preserve=True, hostbuf={}),
               dict(phase_preserve=True, time_map=np.arange(12.0))):
        with pytest.raises(ValueError, match="phase_preserve"):
            ss.synth(rc.SR, 256, **kw)


def test_export_argument_errors():
    """pvk_track_relink checks sizes, npks, pointers and the 2^31 limit before any CUDA call."""
    L = eh.lib()
    tid, pk, _ = run_table(8, 4, seed=2)
    tau = np.array([3.0, 1.5, 0.0])
    tm = tme.time_map(tid, pk, tau)[0]
    to, lo = np.zeros((3, 4), dtype=np.int32), np.zeros((3, 4), dtype=np.int32)
    nto = np.zeros(1, dtype=np.int32)
    wsb = int(L.pvk_track_relink_workspace_bytes(8, 4, 3))
    ws = np.zeros(wsb, dtype=np.uint8)
    nt = len(pk["tstart"])
    assert L.pvk_track_relink_workspace_bytes(-1, 4, 3) == -1 and L.pvk_track_relink_workspace_bytes(8, 0, 3) == -1

    def call(nframes=8, npks=4, ntracks=nt, B=3, tid_p=eh.ptr(tid), tmap=eh.ptr(tau), tid_out=eh.ptr(to),
             ntracks_out=eh.ptr(nto), toff=eh.ptr(pk["toff"]), ws_p=eh.ptr(ws), ws_bytes=wsb):
        return L.pvk_track_relink(tid_p, nframes, npks, ntracks, eh.ptr(pk["tstart"]), eh.ptr(pk["tlen"]), toff,
                                  eh.ptr(tm), tmap, B, tid_out, eh.ptr(lo), ntracks_out, ws_p, ws_bytes, None)
    assert call() == 0 and nto[0] > 0
    assert call(B=0, tid_p=None, tmap=None, tid_out=None, ws_p=None, ws_bytes=0) == 0 and nto[0] == 0
    for kw in (dict(npks=0), dict(npks=1025), dict(nframes=-1), dict(ntracks=-1), dict(B=-1), dict(nframes=0),
               dict(B=1 << 30), dict(tid_p=None), dict(tmap=None), dict(tid_out=None), dict(ntracks_out=None),
               dict(toff=None), dict(ws_p=None), dict(ws_bytes=wsb - 1)):
        assert call(**kw) != 0, kw
        assert b"pvk_track_relink" in L.pvk_last_error()
